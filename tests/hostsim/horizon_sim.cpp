// TEST INFRASTRUCTURE ONLY.  The shadow horizon map (csrc/vrm_core.cuh HorizonView, vrm_flat.cuh FlatRay::past_horizon) on the host:
// hostsim.cpp (the product's traversal compiled for the host, unchanged) plus entry points that build the map the product's way
// (horizon_setup + one horizon_splat per occupied cluster) and hand it to the state machine.  Compiled on demand by tests/horizon_sim.py
// with the flags of tests/hostsim/Makefile.
#include "hostsim.cpp"

namespace {

// The map of s for gLight; cells stay owned by `cells`.  Off (null cells) when the light gets none.
HorizonView horizon_map(const SimScene& s, std::vector<int32_t>& cells)
{
	HorizonView h;
	h.cells = nullptr;
	if (!gLight.useShadows) return h;
	const uint32_t axis0 = (uint32_t)unpack_perm(make_light_walk(gLight).laPerm).a0;
	if (!horizon_setup(gLight.dir, s.diameter, axis0, h)) return h;
	cells.assign((size_t)h.nu * h.nv, kHorizonEmpty);
	const uint32_t D = s.diameter;
	for (size_t t = 0; t < s.regionTable.size(); t++)
	{
		const int32_t ri = s.regionTable[t];
		if (ri < 0) continue;
		const uint32_t ux = (uint32_t)(t % D), uy = (uint32_t)((t / D) % D), uz = (uint32_t)(t / ((size_t)D * D));
		for (uint32_t cid = 0; cid < 512; cid++)
			if ((s.clusterMask[(size_t)ri * 16 + (cid >> 5)] >> (cid & 31u)) & 1u)
				horizon_splat(h, ux * 8 + (cid >> 6), uy * 8 + ((cid >> 3) & 7u), uz * 8 + (cid & 7u),
				              [&](uint32_t i, int32_t v) { if (v > cells[i]) cells[i] = v; });
	}
	h.cells = cells.data();
	return h;
}

// hostsim.cpp's render_rows with the map in every context (counters: nExist, nExistFalse, nLookup, nLookupHit, max nLookup per ray)
template <int ST, int ALGO>
void render_hz(const SimScene& s, const HorizonView hv, const float* cam, const float* tr, float scale, uint32_t W, uint32_t H, uint8_t* rgb,
               int32_t* hits, uint64_t* counters, int nThreads)
{
	uint64_t total[5] = {0, 0, 0, 0, 0};
	#pragma omp parallel num_threads(nThreads)
	{
		RayCtx<ST, true> c;
		c.sv = s.view(); c.light = gLight; c.lw = make_light_walk(gLight); c.hitOut = c.hit;
		c.translation[0] = tr[0]; c.translation[1] = tr[1]; c.translation[2] = tr[2];
		uint64_t local[5] = {0, 0, 0, 0, 0};
		#pragma omp for schedule(dynamic, 1)
		for (int64_t y = 0; y < (int64_t)H; y++)
			for (uint32_t x = 0; x < W; x++)
			{
				float o[3], d[3];
				c.reset();
				c.hv = hv;
				if (gFlat) primary_ray_flat(cam, x, (uint32_t)y, W, H, 1.0f / (float)W, 1.0f / (float)H, o, d);
				else primary_ray(cam, x, (uint32_t)y, W, H, o, d);
				const uint32_t color = march<ST, ALGO>(c, o, d, scale);
				const size_t p = (size_t)y * W + x;
				rgb[3 * p] = (uint8_t)(color >> 16); rgb[3 * p + 1] = (uint8_t)((color >> 8) & 0xFF); rgb[3 * p + 2] = (uint8_t)(color & 0xFF);
				if (hits) memcpy(hits + 4 * p, c.hit, 16);
				local[0] += c.st.nExist; local[1] += c.st.nExistFalse; local[2] += c.st.nLookup; local[3] += c.st.nLookupHit;
				if (c.st.nLookup > local[4]) local[4] = c.st.nLookup;
			}
		#pragma omp critical
		{
			for (int i = 0; i < 4; i++) total[i] += local[i];
			if (local[4] > total[4]) total[4] = local[4];
		}
	}
	if (counters) memcpy(counters, total, sizeof(total));
}

}  // namespace

extern "C" {

// Camera.cuh:11-23 (tools/warp_profile.py: cameras without the GPU library)
void hz_camera_make(const float* origin, const float* lookAt, const float* up, float fov, float aspect, float* out)
{
	auto unit = [](const float* a, float* r) { const float l = sqrtf(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]); r[0] = a[0] / l; r[1] = a[1] / l; r[2] = a[2] / l; };
	auto cross = [](const float* a, const float* b, float* r) { r[0] = a[1] * b[2] - a[2] * b[1]; r[1] = a[2] * b[0] - a[0] * b[2]; r[2] = a[0] * b[1] - a[1] * b[0]; };
	const float halfHeight = tanf((fov * 3.14159265358979323846f / 180.f) / 2.0f), halfWidth = halfHeight * aspect;
	const float dir[3] = {lookAt[0] - origin[0], lookAt[1] - origin[1], lookAt[2] - origin[2]};
	float w[3], wxup[3], u[3], v[3];
	unit(dir, w); cross(w, up, wxup); unit(wxup, u); cross(u, w, v);
	for (int i = 0; i < 3; i++)
	{
		out[i] = origin[i];
		out[3 + i] = origin[i] - halfWidth * u[i] - halfHeight * v[i] + w[i];
		out[6 + i] = (2 * halfWidth) * u[i];
		out[9 + i] = (2 * halfHeight) * v[i];
		out[12 + i] = w[i];
	}
}

// sim_render with the horizon map on (horizon != 0) or off, in the traversal form of sim_set_flat
int hz_render(void* h, const float* cam, const float* tr, uint32_t scale, int algorithm, uint32_t W, uint32_t H, uint8_t* rgb, int32_t* hits,
              uint64_t* counters, int nThreads, int horizon)
{
	SimScene* s = static_cast<SimScene*>(h);
	if (s->storage == -1) return 1;
	if (nThreads < 1) nThreads = 1;
	std::vector<int32_t> cells;
	HorizonView hv;
	hv.cells = nullptr;
	if (horizon) hv = horizon_map(*s, cells);
	const float sc = (float)scale;
	if (s->storage == kStorageHash)
	{
		if (algorithm == kAlgoOriginal) render_hz<kStorageHash, kAlgoOriginal>(*s, hv, cam, tr, sc, W, H, rgb, hits, counters, nThreads);
		else render_hz<kStorageHash, kAlgoLongestAxis>(*s, hv, cam, tr, sc, W, H, rgb, hits, counters, nThreads);
	}
	else
	{
		if (algorithm == kAlgoOriginal) render_hz<kStorageVcs, kAlgoOriginal>(*s, hv, cam, tr, sc, W, H, rgb, hits, counters, nThreads);
		else render_hz<kStorageVcs, kAlgoLongestAxis>(*s, hv, cam, tr, sc, W, H, rgb, hits, counters, nThreads);
	}
	return 0;
}

// Lockstep warp simulation of march_scene_flat_warp's hit barrier (as sim_warp_profile, VCS + longest axis, 8x4 tiles sampled every
// tileStride-th in both directions) with the horizon map on or off.  out: {tiles, passes, shadow-ray passes}
int hz_warp_passes(void* h, const float* cam, const float* tr, uint32_t scale, uint32_t W, uint32_t H, uint32_t tileStride, int horizon,
                   uint64_t* out, int nThreads)
{
	SimScene* s = static_cast<SimScene*>(h);
	if (s->storage != kStorageVcs) return 1;
	using Ray = FlatRay<kStorageVcs, kAlgoLongestAxis, false>;
	std::vector<int32_t> cells;
	HorizonView hv;
	hv.cells = nullptr;
	if (horizon) hv = horizon_map(*s, cells);
	const uint32_t tilesX = (W + 7) / 8, tilesY = (H + 3) / 4;
	uint64_t T[3] = {0, 0, 0};
	#pragma omp parallel num_threads(nThreads)
	{
		uint64_t t[3] = {0, 0, 0};
		RayCtx<kStorageVcs, false> c;
		c.sv = s->view(); c.light = gLight; c.lw = make_light_walk(gLight); c.hitOut = nullptr;
		c.translation[0] = tr[0]; c.translation[1] = tr[1]; c.translation[2] = tr[2];
		c.reset();
		c.skipDead = 1u;
		c.hv = hv;
		#pragma omp for schedule(dynamic, 1)
		for (int64_t ty = 0; ty < (int64_t)tilesY; ty += tileStride)
			for (uint32_t tx = 0; tx < tilesX; tx += tileStride)
			{
				Ray ray[32];
				for (int l = 0; l < 32; l++)
				{
					const uint32_t x = tx * 8 + (l & 7), y = (uint32_t)ty * 4 + (l >> 3);
					ray[l].st = kStDone; ray[l].result = 0;
					if (x < W && y < H)
					{
						float o[3], d[3];
						primary_ray_flat(cam, x, y, W, H, 1.0f / (float)W, 1.0f / (float)H, o, d);
						ray[l].start_primary(c, o, d, (float)scale);
					}
				}
				t[0]++;
				for (;;)
				{
					bool marching = false, anyHit = false, shadowPass = false;
					for (int l = 0; l < 32; l++)
					{
						if (ray[l].st <= kStHead) { marching = true; if (ray[l].shadow()) shadowPass = true; }
						if (ray[l].st == kStHit) anyHit = true;
					}
					if (marching)
					{
						t[1]++;
						if (shadowPass) t[2]++;
						for (int l = 0; l < 32; l++) if (ray[l].st <= kStHead) ray[l].template step_marching<kPpOff>(c);
						continue;
					}
					if (!anyHit) break;
					for (int l = 0; l < 32; l++) if (ray[l].st == kStHit) ray[l].do_hit(c);
				}
			}
		#pragma omp critical
		for (int i = 0; i < 3; i++) T[i] += t[i];
	}
	memcpy(out, T, sizeof(T));
	return 0;
}

// Property of the map (tests/test_shadow_horizon.py): trace the given primary rays (VCS, generic state machine) to their hits, start each
// hit's shadow ray WITHOUT the early exit and march it in full; the threshold horizon_threshold() gives it must never be passed at the end
// of a step whose voxel test found an occupied cluster.  out: {shadow rays, violations, rays that walked past their threshold, voxel tests
// of shadow rays that found an occupied cluster}.  Returns 1 when the light gets no map.
int hz_property(void* h, const float* rays, uint64_t n, int algorithm, uint64_t* out)
{
	SimScene* s = static_cast<SimScene*>(h);
	if (s->storage != kStorageVcs) return 2;
	std::vector<int32_t> cells;
	const HorizonView hv = horizon_map(*s, cells);
	if (!hv.cells) return 1;
	auto run = [&](auto tag) {
		using Ray = decltype(tag);
		uint64_t t[4] = {0, 0, 0, 0};
		RayCtx<kStorageVcs, true> c;
		c.sv = s->view(); c.light = gLight; c.lw = make_light_walk(gLight); c.hitOut = nullptr;
		c.translation[0] = c.translation[1] = c.translation[2] = 0.0f;
		for (uint64_t i = 0; i < n; i++)
		{
			c.reset();
			Ray ray;
			ray.start_primary(c, rays + 6 * i, rays + 6 * i + 3, 1.0f);
			while (ray.st <= kStHead) ray.template step_marching<kPpInline>(c);
			if (ray.st != kStHit) continue;
			ShadowStart ss;
			ray.shade_hit(c, ss);
			ray.start_shadow(c, ss);  // (c.hv.cells null: no early exit)
			RayCtx<kStorageVcs, true> cm = c;
			cm.hv = hv;
			const int32_t thr = ray.horizon_threshold(cm, ss);
			t[0]++;
			bool passed = false;
			while (ray.st <= kStHead)
			{
				const unsigned long long found = c.st.nExist - c.st.nExistFalse;
				ray.template step_marching<kPpInline>(c);
				Ray probe = ray;
				probe.fl = (probe.fl & ((1u << kFlHzShift) - 1u)) | ((uint32_t)thr << kFlHzShift);
				const bool past = probe.past_horizon();
				if (c.st.nExist - c.st.nExistFalse > found) { t[3]++; if (past) t[1]++; }
				passed = passed || past;
			}
			if (passed) t[2]++;
		}
		memcpy(out, t, sizeof(t));
	};
	if (algorithm == kAlgoOriginal) run(FlatRay<kStorageVcs, kAlgoOriginal, true>());
	else run(FlatRay<kStorageVcs, kAlgoLongestAxis, true>());
	return 0;
}

}  // extern "C"
