// TEST INFRASTRUCTURE ONLY.  The exact ray cast (csrc/vrm_core.cuh cast_ray, the source the sm_100a kernel of csrc/vrm_cast.cu is built
// from) on the host: hostsim.cpp (its naive builder fills both storage layouts, unchanged) plus entry points for rays and views.  Compiled
// on demand by tests/cast_ref.py with the flags of tests/hostsim/Makefile.
#include "hostsim.cpp"

namespace {

void cast_one(const SimScene& s, const float* P, const float* D, const float* tr, float scale, float tNear, float tFar, float len, bool withLen,
              int32_t* hit, float* depth, uint8_t* face, uint32_t* colour)
{
	CastResult r;
	const SceneView sv = s.view();
	if (s.storage == kStorageHash) cast_ray<kStorageHash>(sv, P, D, tr, scale, tNear, tFar, len, withLen, r);
	else cast_ray<kStorageVcs>(sv, P, D, tr, scale, tNear, tFar, len, withLen, r);
	memcpy(hit, r.hit, 16);
	*depth = r.depth;
	*face = (uint8_t)r.face;
	*colour = r.colour;
}

}  // namespace

extern "C" {

// rays = n x 6 floats, ranges = n x 2 {t_near, t_far} or NULL for [0, +inf)
int cast_rays(void* h, const float* rays, const float* ranges, uint64_t n, const float* tr, uint32_t scale, int32_t* hits, float* depth,
              uint8_t* face, uint32_t* colour)
{
	const SimScene* s = static_cast<SimScene*>(h);
	if (s->storage == -1) return 1;
	#pragma omp parallel for schedule(dynamic, 256)
	for (int64_t i = 0; i < (int64_t)n; i++)
		cast_one(*s, rays + 6 * i, rays + 6 * i + 3, tr, (float)scale, ranges ? ranges[2 * i] : 0.0f, ranges ? ranges[2 * i + 1] : INFINITY, 0.0f,
		         false, hits + 4 * i, depth + i, face + i, colour + i);
	return 0;
}

// cameras = n_views x 15 floats; outputs view-major, n_views x H x W
int cast_views(void* h, const float* cameras, uint32_t nViews, const float* tr, uint32_t scale, uint32_t W, uint32_t H, int32_t* hits, float* depth,
               uint8_t* face, uint32_t* colour)
{
	const SimScene* s = static_cast<SimScene*>(h);
	if (s->storage == -1) return 1;
	const int64_t px = (int64_t)W * H;
	#pragma omp parallel for schedule(dynamic, 64)
	for (int64_t i = 0; i < (int64_t)nViews * px; i++)
	{
		const uint32_t v = (uint32_t)(i / px), y = (uint32_t)((i % px) / W), x = (uint32_t)(i % W);
		float P[3], D[3], len;
		primary_ray(cameras + 15 * (size_t)v, x, y, W, H, P, D, len);
		cast_one(*s, P, D, tr, (float)scale, 0.0f, INFINITY, len, true, hits + 4 * i, depth + i, face + i, colour + i);
	}
	return 0;
}

}  // extern "C"
