// vrm_cast.cu -- exact ray casts through a built scene (include/vrm_b200.h, "exact ray casts"; DESIGN.md §3.7).
//
// One thread per ray (or pixel) in caller order, running vrm_core.cuh cast_ray, the one definition the CPU tests also compile.  The hit record
// leaves as one 16-byte store; depth, face and colour element by element.  Every output is nullable.
#include "vrm_internal.h"
#include "../../include/vrm_b200.h"

using namespace vrm;

namespace
{

constexpr int kThreads = 128;
constexpr uint64_t kMaxRecords = 1ull << 37;  // 2 TiB of hit records: far beyond any device, keeps the grid below 2^31 blocks

struct CastArgs
{
	SceneView sv;
	const float* rays;    // rays: n x 6 floats; views: null
	const float* ranges;  // rays: n x 2 {t_near, t_far}, null = [0, +inf)
	const float* cams;    // views: n_views x 15 floats in device memory; null when `cam` holds the only view
	float cam[VRM_CAMERA_FLOATS];
	float tr[3];
	float scale;
	uint32_t W, H;
	uint64_t n;
	int4* hits;
	float* depth;
	uint8_t* face;
	uint32_t* colour;
};

template <int ST, bool VIEWS>
__global__ void __launch_bounds__(kThreads) cast_kernel(const __grid_constant__ CastArgs a)
{
	const uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x;
	if (i >= a.n) return;
	float P[3], D[3], len = 0.0f, tNear = 0.0f, tFar = INFINITY;
	if constexpr (VIEWS)
	{
		const uint64_t px = (uint64_t)a.W * a.H;
		const uint32_t v = (uint32_t)(i / px);
		const uint64_t p = i - (uint64_t)v * px;
		const uint32_t y = (uint32_t)(p / a.W), x = (uint32_t)(p - (uint64_t)y * a.W);
		primary_ray(a.cams ? a.cams + (size_t)v * VRM_CAMERA_FLOATS : a.cam, x, y, a.W, a.H, P, D, len);
	}
	else
	{
		const float* r = a.rays + 6 * i;
		for (int c = 0; c < 3; c++) { P[c] = __ldg(r + c); D[c] = __ldg(r + 3 + c); }
		if (a.ranges) { tNear = __ldg(a.ranges + 2 * i); tFar = __ldg(a.ranges + 2 * i + 1); }
	}
	CastResult res;
	cast_ray<ST>(a.sv, P, D, a.tr, a.scale, tNear, tFar, len, VIEWS, res);
	if (a.hits) a.hits[i] = make_int4(res.hit[0], res.hit[1], res.hit[2], res.hit[3]);
	if (a.depth) a.depth[i] = res.depth;
	if (a.face) a.face[i] = (uint8_t)res.face;
	if (a.colour) a.colour[i] = res.colour;
}

int launch_cast(vrm_scene* s, uint64_t n, const float* d_rays, const float* d_ranges, const float* d_cams, const float* h_cam, uint32_t W, uint32_t H,
                const float* translation, uint32_t scale, int32_t* d_hits, float* d_depth, uint8_t* d_face, uint32_t* d_colour)
{
	CastArgs a = {};
	a.sv = s->view();
	a.rays = d_rays; a.ranges = d_ranges; a.cams = d_cams;
	if (h_cam) for (int i = 0; i < VRM_CAMERA_FLOATS; i++) a.cam[i] = h_cam[i];
	for (int i = 0; i < 3; i++) a.tr[i] = translation[i];
	a.scale = (float)scale;
	a.W = W; a.H = H; a.n = n;
	a.hits = reinterpret_cast<int4*>(d_hits); a.depth = d_depth; a.face = d_face; a.colour = d_colour;
	const uint64_t blocks = (n + kThreads - 1) / kThreads;  // < 2^31 (kMaxRecords)
	const bool views = d_rays == nullptr;
	if (s->storage == kStorageHash)
	{
		if (views) cast_kernel<kStorageHash, true><<<(unsigned)blocks, kThreads, 0, s->stream>>>(a);
		else cast_kernel<kStorageHash, false><<<(unsigned)blocks, kThreads, 0, s->stream>>>(a);
	}
	else
	{
		if (views) cast_kernel<kStorageVcs, true><<<(unsigned)blocks, kThreads, 0, s->stream>>>(a);
		else cast_kernel<kStorageVcs, false><<<(unsigned)blocks, kThreads, 0, s->stream>>>(a);
	}
	VRM_CUDA(s, cudaGetLastError());
	return VRM_OK;
}

// Checks shared by the four entry points.  Returns -1 when the call goes on, else the status to return (VRM_OK for zero records).
int check_cast(vrm_scene* s, uint64_t n, const void* src, const float* translation, uint32_t scale, const int32_t* hits, const float* depth,
               const uint8_t* face, const uint32_t* colour, bool device)
{
	if (!s) return VRM_ERR_INVALID;
	if (s->storage < 0) { s->lastError = "cast: the scene is not built"; return VRM_ERR_STATE; }
	if (!translation) { s->lastError = "cast: translation is NULL"; return VRM_ERR_INVALID; }
	if (scale == 0) { s->lastError = "cast: scale is 0"; return VRM_ERR_INVALID; }
	if (!hits && !depth && !face && !colour) { s->lastError = "cast: every output is NULL"; return VRM_ERR_INVALID; }
	if (n == 0) return VRM_OK;
	if (!src) { s->lastError = "cast: rays or cameras is NULL"; return VRM_ERR_INVALID; }
	if (n > kMaxRecords) { s->lastError = "cast: more than 2^37 records"; return VRM_ERR_INVALID; }
	if (device && ((reinterpret_cast<uintptr_t>(hits) & 15u) || (reinterpret_cast<uintptr_t>(depth) & 3u) || (reinterpret_cast<uintptr_t>(colour) & 3u)))
	{ s->lastError = "cast: device hits must be 16-byte aligned, device depth and colour 4-byte aligned"; return VRM_ERR_INVALID; }
	return -1;
}

// Host outputs are staged in one device buffer: [hits 16n][depth 4n][colour 4n][face n], each part only when asked for.
struct Staged
{
	int32_t* hits; float* depth; uint32_t* colour; uint8_t* face;
};

int stage_outputs(vrm_scene* s, uint64_t n, size_t inputBytes, bool hits, bool depth, bool colour, bool face, Staged& o, char*& inputs)
{
	const size_t hb = hits ? n * 16 : 0, db = depth ? n * 4 : 0, cb = colour ? n * 4 : 0, fb = face ? n : 0;
	const size_t ib = (inputBytes + 15) & ~size_t(15);
	int rc = vrm_ensure(s, &s->d_io, &s->ioBytes, ib + hb + db + cb + fb);
	if (rc) return rc;
	char* base = static_cast<char*>(s->d_io);
	inputs = base;
	base += ib;
	o.hits = hits ? reinterpret_cast<int32_t*>(base) : nullptr; base += hb;
	o.depth = depth ? reinterpret_cast<float*>(base) : nullptr; base += db;
	o.colour = colour ? reinterpret_cast<uint32_t*>(base) : nullptr; base += cb;
	o.face = face ? reinterpret_cast<uint8_t*>(base) : nullptr;
	return VRM_OK;
}

int copy_back(vrm_scene* s, uint64_t n, const Staged& o, int32_t* hits, float* depth, uint8_t* face, uint32_t* colour)
{
	if (hits) VRM_CUDA(s, cudaMemcpyAsync(hits, o.hits, n * 16, cudaMemcpyDeviceToHost, s->stream));
	if (depth) VRM_CUDA(s, cudaMemcpyAsync(depth, o.depth, n * 4, cudaMemcpyDeviceToHost, s->stream));
	if (colour) VRM_CUDA(s, cudaMemcpyAsync(colour, o.colour, n * 4, cudaMemcpyDeviceToHost, s->stream));
	if (face) VRM_CUDA(s, cudaMemcpyAsync(face, o.face, n, cudaMemcpyDeviceToHost, s->stream));
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	return VRM_OK;
}

int cast_rays(vrm_scene* s, const float* rays, const float* ranges, uint64_t n, const float* translation, uint32_t scale, int32_t* hits, float* depth,
              uint8_t* face, uint32_t* colour, bool device)
{
	int rc = check_cast(s, n, rays, translation, scale, hits, depth, face, colour, device);
	if (rc >= 0) return rc;
	if (device && ((reinterpret_cast<uintptr_t>(rays) & 3u) || (reinterpret_cast<uintptr_t>(ranges) & 3u)))
	{ s->lastError = "cast: device rays and ranges must be 4-byte aligned"; return VRM_ERR_INVALID; }
	VRM_CUDA(s, cudaSetDevice(s->device));
	vrm_apply_l2_window(s);
	if (device) return launch_cast(s, n, rays, ranges, nullptr, nullptr, 0, 0, translation, scale, hits, depth, face, colour);
	const size_t rayBytes = n * 24, rangeBytes = ranges ? n * 8 : 0;
	Staged o;
	char* in;
	rc = stage_outputs(s, n, rayBytes + rangeBytes, hits, depth, colour, face, o, in);
	if (rc) return rc;
	float* d_rays = reinterpret_cast<float*>(in);
	float* d_ranges = ranges ? reinterpret_cast<float*>(in + rayBytes) : nullptr;
	VRM_CUDA(s, cudaMemcpyAsync(d_rays, rays, rayBytes, cudaMemcpyHostToDevice, s->stream));
	if (ranges) VRM_CUDA(s, cudaMemcpyAsync(d_ranges, ranges, rangeBytes, cudaMemcpyHostToDevice, s->stream));
	rc = launch_cast(s, n, d_rays, d_ranges, nullptr, nullptr, 0, 0, translation, scale, o.hits, o.depth, o.face, o.colour);
	if (rc) return rc;
	return copy_back(s, n, o, hits, depth, face, colour);
}

// records of a view batch, 0 when a factor is 0; kMaxRecords + 1 when the product exceeds kMaxRecords
uint64_t view_records(uint32_t nViews, uint32_t W, uint32_t H)
{
	const uint64_t px = (uint64_t)W * H;
	if (px == 0 || nViews == 0) return 0;
	return px > kMaxRecords / nViews ? kMaxRecords + 1 : px * nViews;
}

int cast_views(vrm_scene* s, const float* cameras, uint32_t nViews, const float* translation, uint32_t scale, uint32_t W, uint32_t H, int32_t* hits,
               float* depth, uint8_t* face, uint32_t* colour, bool device)
{
	const uint64_t n = view_records(nViews, W, H);
	int rc = check_cast(s, n, cameras, translation, scale, hits, depth, face, colour, device);
	if (rc >= 0) return rc;
	VRM_CUDA(s, cudaSetDevice(s->device));
	vrm_apply_l2_window(s);
	const bool inlineCam = nViews == 1;  // a single view travels in the kernel arguments
	if (!inlineCam) { rc = vrm_upload_cameras(s, cameras, nViews); if (rc) return rc; }
	const float* d_cams = inlineCam ? nullptr : s->d_cams;
	const float* h_cam = inlineCam ? cameras : nullptr;
	if (device) return launch_cast(s, n, nullptr, nullptr, d_cams, h_cam, W, H, translation, scale, hits, depth, face, colour);
	Staged o;
	char* in;
	rc = stage_outputs(s, n, 0, hits, depth, colour, face, o, in);
	if (rc) return rc;
	rc = launch_cast(s, n, nullptr, nullptr, d_cams, h_cam, W, H, translation, scale, o.hits, o.depth, o.face, o.colour);
	if (rc) return rc;
	return copy_back(s, n, o, hits, depth, face, colour);
}

}  // namespace

extern "C" {

int vrm_cast_rays(vrm_scene* s, const float* rays, const float* ranges, uint64_t n, const float translation[3], uint32_t scale, int32_t* hits_out,
                  float* depth_out, uint8_t* face_out, uint32_t* colour_out)
{
	return cast_rays(s, rays, ranges, n, translation, scale, hits_out, depth_out, face_out, colour_out, false);
}

int vrm_cast_rays_device(vrm_scene* s, const float* d_rays, const float* d_ranges, uint64_t n, const float translation[3], uint32_t scale,
                         int32_t* d_hits_out, float* d_depth_out, uint8_t* d_face_out, uint32_t* d_colour_out)
{
	return cast_rays(s, d_rays, d_ranges, n, translation, scale, d_hits_out, d_depth_out, d_face_out, d_colour_out, true);
}

int vrm_cast_views(vrm_scene* s, const float* cameras, uint32_t n_views, const float translation[3], uint32_t scale, uint32_t width, uint32_t height,
                   int32_t* hits_out, float* depth_out, uint8_t* face_out, uint32_t* colour_out)
{
	return cast_views(s, cameras, n_views, translation, scale, width, height, hits_out, depth_out, face_out, colour_out, false);
}

int vrm_cast_views_device(vrm_scene* s, const float* cameras, uint32_t n_views, const float translation[3], uint32_t scale, uint32_t width,
                          uint32_t height, int32_t* d_hits_out, float* d_depth_out, uint8_t* d_face_out, uint32_t* d_colour_out)
{
	return cast_views(s, cameras, n_views, translation, scale, width, height, d_hits_out, d_depth_out, d_face_out, d_colour_out, true);
}

}  // extern "C"
