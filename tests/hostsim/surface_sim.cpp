// TEST INFRASTRUCTURE ONLY.  The hit-surface definition (csrc/vrm_core.cuh primary_ray + hit_surface, the source the sm_100a kernel of
// csrc/vrm_surface.cu is built from) compiled for the host, record by record, so that the CPU tier can check it against a numpy
// restatement.  Compiled on demand by tests/surface_ref.py with the flags of tests/hostsim/Makefile.
#include <stdint.h>

struct uint2 { uint32_t x, y; };  // the CUDA vector types vrm_core.cuh names
struct uint4 { uint32_t x, y, z, w; };

#include "../../voxelraymarcher_b200/csrc/vrm_core.cuh"

using namespace vrm;

extern "C" {

// hits = n_views x H x W x 4 int32 (view-major), cameras = n_views x 15 floats
void surf_views(const float* cameras, uint32_t nViews, const float* tr, uint32_t scale, uint32_t W, uint32_t H, const int32_t* hits, float* depth,
                uint8_t* face)
{
	uint64_t i = 0;
	for (uint32_t v = 0; v < nViews; v++)
		for (uint32_t y = 0; y < H; y++)
			for (uint32_t x = 0; x < W; x++, i++)
			{
				float P[3] = {0.0f, 0.0f, 0.0f}, D[3] = {0.0f, 0.0f, 0.0f}, len = 0.0f;
				if (hits[4 * i + 3] != 0) primary_ray(cameras + 15 * (size_t)v, x, y, W, H, P, D, len);
				uint32_t f;
				depth[i] = hit_surface(hits + 4 * i, P, D, tr, (float)scale, len, true, f);
				face[i] = (uint8_t)f;
			}
}

// rays = n x 6 floats, hits = n x 4 int32
void surf_rays(const float* rays, uint64_t n, const float* tr, uint32_t scale, const int32_t* hits, float* depth, uint8_t* face)
{
	for (uint64_t i = 0; i < n; i++)
	{
		uint32_t f;
		depth[i] = hit_surface(hits + 4 * i, rays + 6 * i, rays + 6 * i + 3, tr, (float)scale, 0.0f, false, f);
		face[i] = (uint8_t)f;
	}
}

// the pixel rays of a frame as (P, D) = n x 6 floats and their len, for tracing them through vrm_trace_rays
void surf_pixel_rays(const float* camera, uint32_t W, uint32_t H, float* rays, float* len)
{
	uint64_t i = 0;
	for (uint32_t y = 0; y < H; y++)
		for (uint32_t x = 0; x < W; x++, i++) primary_ray(camera, x, y, W, H, rays + 6 * i, rays + 6 * i + 3, len[i]);
}

}  // extern "C"
