// vrm_generate.cu -- procedural scenes generated ON THE GPU straight into a scene's staging list (SURVEY.md §8f-3): the
// voxels of the BASELINE.json workloads never exist on the host, so building a 32 M voxel scene no longer starts with
// seconds of numpy and a 512 MB host-to-device copy.
//
// The generators are the integer-only definitions of voxelraymarcher_b200/scenes.py (terrain: 4-octave fixed-point value
// noise height field; sparse_shells: hashed sphere shells on a coarse lattice) -- same hashes, same arithmetic, so the
// voxel SET and every colour are identical to the host generator's (tests/test_parity_gpu.py builds both and compares).
// Neither scene has duplicate coordinates, so the order inside the staging chunk is irrelevant to the built structure.
#include "vrm_internal.h"
#include "../../include/vrm_b200.h"

namespace
{

constexpr int kThreads = 256;

__host__ __device__ inline uint32_t hash2(uint32_t ix, uint32_t iz, uint32_t seed)  // scenes._hash2
{
	uint32_t h = (ix * 0x9E3779B1u) ^ (iz * 0x85EBCA77u) ^ (seed * 0xC2B2AE3Du);
	h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12; h *= 0x297A2D39u; h ^= h >> 15;
	return h & 0xFFFFu;
}

__host__ __device__ inline uint32_t hash3(uint32_t ix, uint32_t iy, uint32_t iz, uint32_t seed)  // scenes._hash3
{
	uint32_t h = (ix * 0x9E3779B1u) ^ (iy * 0x7FEB352Du) ^ (iz * 0x85EBCA77u) ^ (seed * 0xC2B2AE3Du);
	h ^= h >> 16; h *= 0x21F0AAADu; h ^= h >> 15; h *= 0x735A2D97u; h ^= h >> 15;
	return h;
}

// scenes.terrain_heights + the clip of scenes.terrain: one thread per (x, z) column
__global__ void terrain_heights_kernel(uint32_t size, uint32_t seed, uint32_t maxHeight, uint32_t* __restrict__ heights)
{
	const uint64_t col = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (col >= (uint64_t)size * size) return;
	const uint32_t x = (uint32_t)(col / size), z = (uint32_t)(col % size);
	const uint32_t amps[4] = {96, 48, 24, 12}, lattices[4] = {128, 64, 32, 16};
	long long h = 32ll << 16;
	for (int o = 0; o < 4; o++)
	{
		const uint32_t lat = lattices[o], s = seed + (uint32_t)o;
		const uint32_t ix = x / lat, iz = z / lat;
		const long long fx = (long long)((x % lat) * 256u / lat), fz = (long long)((z % lat) * 256u / lat);  // 8-bit fractions
		const long long v00 = hash2(ix, iz, s), v10 = hash2(ix + 1, iz, s), v01 = hash2(ix, iz + 1, s), v11 = hash2(ix + 1, iz + 1, s);
		const long long top = v00 * (256 - fx) + v10 * fx, bot = v01 * (256 - fx) + v11 * fx;
		h += (long long)amps[o] * ((top * (256 - fz) + bot * fz) >> 16);
	}
	long long v = h >> 16;
	const long long hi = (long long)maxHeight - 1;
	v = v < 1 ? 1 : (v > hi ? hi : v);
	heights[col] = (uint32_t)v;
}

__device__ inline uint32_t height_colour(uint32_t y)  // scenes._height_colour
{
	const uint32_t r = y < 40 ? 194u : (y < 90 ? 60u : (y < 140 ? 120u : 240u));
	const uint32_t g = y < 40 ? 178u : (y < 90 ? 160u : (y < 140 ? 120u : 240u));
	const uint32_t b = y < 40 ? 128u : (y < 90 ? 70u : (y < 140 ? 125u : 250u));
	const uint32_t shade = (y % 8u) * 2u;
	return ((r - shade) << 16) | ((g - shade) << 8) | (b - shade);
}

// One thread per voxel: the column is found by binary search in the exclusive scan of the heights (columns are x-major,
// voxels of a column bottom-up: the order of scenes.terrain).
__global__ void terrain_fill_kernel(uint32_t size, const uint32_t* __restrict__ starts, uint64_t total, int32_t* __restrict__ xyz, uint32_t* __restrict__ rgb)
{
	const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (i >= total) return;
	uint32_t lo = 0, hi = size * size;  // last column with starts[col] <= i
	while (hi - lo > 1)
	{
		const uint32_t mid = lo + (hi - lo) / 2;
		if ((uint64_t)starts[mid] <= i) lo = mid; else hi = mid;
	}
	const uint32_t y = (uint32_t)(i - starts[lo]);
	xyz[3 * i] = (int32_t)(lo / size); xyz[3 * i + 1] = (int32_t)y; xyz[3 * i + 2] = (int32_t)(lo % size);
	rgb[i] = height_colour(y);
}

// scenes.sparse_shells: number of lattice points with (r-1)^2 <= d^2 < r^2, one block per radius
__global__ void shell_count_kernel(uint32_t* __restrict__ counts)
{
	const int r = (int)blockIdx.x;
	const int w = 2 * r + 1;
	uint32_t mine = 0;
	for (int t = (int)threadIdx.x; t < w * w * w; t += (int)blockDim.x)
	{
		const int x = t / (w * w) - r, y = (t / w) % w - r, z = t % w - r;
		const int d2 = x * x + y * y + z * z;
		if (d2 < r * r && d2 >= (r - 1) * (r - 1)) mine++;
	}
	__shared__ uint32_t total;
	if (threadIdx.x == 0) total = 0;
	__syncthreads();
	atomicAdd(&total, mine);
	__syncthreads();
	if (threadIdx.x == 0) counts[r] = total;
}

__device__ inline bool shell_of_cell(uint32_t cell, uint32_t n, uint32_t cellSize, uint32_t seed, uint32_t fillPct, uint32_t& h, uint32_t& r)
{
	const uint32_t cx = cell / (n * n), cy = (cell / n) % n, cz = cell % n;
	h = hash3(cx, cy, cz, seed);
	r = cellSize / 8u + ((h >> 8) % (cellSize / 4u));
	return (h % 100u) < fillPct;
}

__global__ void shell_cells_kernel(uint32_t n, uint32_t cellSize, uint32_t seed, uint32_t fillPct, const uint32_t* __restrict__ shellCounts, uint32_t* __restrict__ cellCounts)
{
	const uint64_t cell = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (cell >= (uint64_t)n * n * n) return;
	uint32_t h, r;
	cellCounts[cell] = shell_of_cell((uint32_t)cell, n, cellSize, seed, fillPct, h, r) ? shellCounts[r] : 0u;
}

// one block per lattice cell
__global__ void shell_fill_kernel(uint32_t n, uint32_t cellSize, uint32_t seed, uint32_t fillPct, const uint32_t* __restrict__ starts,
                                  int32_t* __restrict__ xyz, uint32_t* __restrict__ rgb)
{
	const uint32_t cell = blockIdx.x;
	uint32_t h, ur;
	if (!shell_of_cell(cell, n, cellSize, seed, fillPct, h, ur)) return;
	const int r = (int)ur, w = 2 * r + 1;
	const int cx = (int)(cell / (n * n)), cy = (int)((cell / n) % n), cz = (int)(cell % n);
	const int ox = cx * (int)cellSize + (int)cellSize / 2, oy = cy * (int)cellSize + (int)cellSize / 2, oz = cz * (int)cellSize + (int)cellSize / 2;
	const uint32_t colour = ((64u + (h & 127u)) << 16) | ((64u + ((h >> 7) & 127u)) << 8) | (64u + ((h >> 14) & 127u));
	__shared__ uint32_t cursor;
	if (threadIdx.x == 0) cursor = 0;
	__syncthreads();
	const uint64_t base = starts[cell];
	for (int t = (int)threadIdx.x; t < w * w * w; t += (int)blockDim.x)
	{
		const int x = t / (w * w) - r, y = (t / w) % w - r, z = t % w - r;
		const int d2 = x * x + y * y + z * z;
		if (d2 < r * r && d2 >= (r - 1) * (r - 1))
		{
			const uint64_t i = base + atomicAdd(&cursor, 1u);
			xyz[3 * i] = ox + x; xyz[3 * i + 1] = oy + y; xyz[3 * i + 2] = oz + z;
			rgb[i] = colour;
		}
	}
}

// The reference's own (host-loop) generators, geometry/VoxelCube.cuh:10-39 and VoxelSphere.cuh:10-66, as index -> voxel maps
// in the reference's INSERTION ORDER (faces of a cube overlap on its edges and shapes may overlap each other: the last
// insert wins, so the order inside the staging chunk is part of the result).
__global__ void cube_kernel(int xp, int yp, int zp, int hw, int32_t* __restrict__ xyz, uint32_t* __restrict__ rgb)
{
	const uint64_t w = 2ull * (uint64_t)hw, perGroup = 2ull * w * w;
	const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (i >= 3ull * perGroup) return;
	const int group = (int)(i / perGroup);           // 0: the two z faces (red), 1: x faces (green), 2: y faces (blue)
	const uint64_t j = i % perGroup, pair = j / 2;
	const bool second = (j & 1ull) != 0;
	const int a = (int)(pair / w) - hw, b = (int)(pair % w) - hw;  // outer / inner loop variable
	int x, y, z;
	uint32_t colour;
	if (group == 0) { x = xp + a; y = yp + b; z = zp + (second ? -hw : hw); colour = 0xFF0000u; }
	else if (group == 1) { x = xp + (second ? hw : -hw); y = yp + a; z = zp + b; colour = 0x00FF00u; }
	else { x = xp + a; y = yp + (second ? hw : -hw); z = zp + b; colour = 0x0000FFu; }
	xyz[3 * i] = x; xyz[3 * i + 1] = y; xyz[3 * i + 2] = z;
	rgb[i] = colour;
}

// candidate index (x-major, then y, then z) -> lattice point of the shell's bounding cube; all arithmetic uint32 as in the reference
__device__ inline bool sphere_point(uint64_t idx, uint32_t xp, uint32_t yp, uint32_t zp, uint32_t r, uint32_t step, uint32_t& x, uint32_t& y, uint32_t& z)
{
	const uint32_t n = 2u * r;
	const uint32_t ix = (uint32_t)(idx / ((uint64_t)n * n)), iy = (uint32_t)((idx / n) % n), iz = (uint32_t)(idx % n);
	x = xp - r + ix * step; y = yp - r + iy; z = zp - r + iz;
	const uint32_t d2 = (x - xp) * (x - xp) + (y - yp) * (y - yp) + (z - zp) * (z - zp);
	return d2 < r * r && d2 > (r - 1u) * (r - 1u);
}

__global__ void sphere_flag_kernel(uint32_t xp, uint32_t yp, uint32_t zp, uint32_t r, uint32_t step, uint64_t candidates, uint32_t* __restrict__ flags)
{
	const uint64_t idx = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (idx >= candidates) return;
	uint32_t x, y, z;
	flags[idx] = sphere_point(idx, xp, yp, zp, r, step, x, y, z) ? 1u : 0u;
}

__global__ void sphere_fill_kernel(uint32_t xp, uint32_t yp, uint32_t zp, uint32_t r, uint32_t step, uint64_t candidates, const uint32_t* __restrict__ pos,
                                   int32_t* __restrict__ xyz, uint32_t* __restrict__ rgb)
{
	const uint64_t idx = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (idx >= candidates) return;
	uint32_t x, y, z;
	if (!sphere_point(idx, xp, yp, zp, r, step, x, y, z)) return;
	const uint32_t xMin = xp - r, xMax = xp + r, yMin = yp - r, yMax = yp + r, zMin = zp - r;
	// the reference's colour ramp, quirks included: green measures y from xMin and the blue divisor is xMax - zMin
	const uint32_t red = 50u + (x - xMin) * (200u / (xMax - xMin));
	const uint32_t green = 50u + (y - xMin) * (200u / (yMax - yMin));
	const uint32_t blue = 50u + (z - zMin) * (200u / (xMax - zMin));
	const uint64_t o = pos[idx];
	xyz[3 * o] = (int32_t)x; xyz[3 * o + 1] = (int32_t)y; xyz[3 * o + 2] = (int32_t)z;
	rgb[o] = (min(red, 255u) << 16) | (min(green, 255u) << 8) | min(blue, 255u);
}

struct Buf
{
	void* p = nullptr;
	~Buf() { if (p) cudaFree(p); }
	template <class T> T* as() { return static_cast<T*>(p); }
};

// exclusive scan of counts[0..n) into starts[0..n], total returned through the host
int scan_counts(vrm_scene* s, const uint32_t* counts, uint32_t* starts, uint64_t n, uint64_t* total)
{
	Buf scratch;
	VRM_CUDA(s, cudaMalloc(&scratch.p, vrm_scan_scratch_elems(n) * 4));
	vrm_exclusive_scan_u32(counts, starts, n, scratch.as<uint32_t>(), s->stream);
	uint32_t last[2] = {0, 0};
	VRM_CUDA(s, cudaMemcpyAsync(&last[0], starts + (n - 1), 4, cudaMemcpyDeviceToHost, s->stream));
	VRM_CUDA(s, cudaMemcpyAsync(&last[1], counts + (n - 1), 4, cudaMemcpyDeviceToHost, s->stream));
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	*total = (uint64_t)last[0] + last[1];
	return VRM_OK;
}

int check_generate(vrm_scene* s)
{
	if (!s) return VRM_ERR_INVALID;
	if (int rc = vrm_check_staging(s)) return rc;
	VRM_CUDA(s, cudaSetDevice(s->device));
	return VRM_OK;
}

unsigned grid_for(uint64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

}  // namespace

extern "C" {

int vrm_scene_generate_terrain(vrm_scene* s, uint32_t size, uint32_t seed, uint32_t max_height, uint64_t* n_out)
{
	int rc = check_generate(s);
	if (rc) return rc;
	if (size < 2 || size > 4096) { s->lastError = "terrain size must be in [2, 4096]"; return VRM_ERR_INVALID; }
	if (max_height == 0) max_height = size;
	if (max_height < 2) { s->lastError = "terrain max_height must be at least 2"; return VRM_ERR_INVALID; }
	const uint64_t cols = (uint64_t)size * size;
	Buf heights, starts;
	VRM_CUDA(s, cudaMalloc(&heights.p, cols * 4));
	VRM_CUDA(s, cudaMalloc(&starts.p, cols * 4));
	terrain_heights_kernel<<<grid_for(cols), kThreads, 0, s->stream>>>(size, seed, max_height, heights.as<uint32_t>());
	uint64_t total = 0;
	rc = scan_counts(s, heights.as<uint32_t>(), starts.as<uint32_t>(), cols, &total);
	if (rc) return rc;
	if (total >= (1ull << 32)) { s->lastError = "terrain has more than 2^32 voxels"; return VRM_ERR_INVALID; }
	int32_t* d_xyz = nullptr; uint32_t* d_rgb = nullptr;
	rc = vrm_stage_reserve(s, total, &d_xyz, &d_rgb);  // appended to the scene's staging arrays, in insertion order
	if (rc) return rc;
terrain_fill_kernel<<<grid_for(total), kThreads, 0, s->stream>>>(size, starts.as<uint32_t>(), total, d_xyz, d_rgb);
	VRM_CUDA(s, cudaGetLastError());
	rc = vrm_stage_commit(s, total);
	if (rc) return rc;
	if (n_out) *n_out = total;
	return VRM_OK;
}

int vrm_scene_generate_cube(vrm_scene* s, int32_t x, int32_t y, int32_t z, int32_t half_width, uint64_t* n_out)
{
	int rc = check_generate(s);
	if (rc) return rc;
	if (half_width < 1 || half_width > 4096) { s->lastError = "cube half width must be in [1, 4096]"; return VRM_ERR_INVALID; }
	const uint64_t w = 2ull * (uint64_t)half_width, total = 6ull * w * w;
	int32_t* d_xyz = nullptr; uint32_t* d_rgb = nullptr;
	rc = vrm_stage_reserve(s, total, &d_xyz, &d_rgb);  // appended to the scene's staging arrays, in insertion order
	if (rc) return rc;
cube_kernel<<<grid_for(total), kThreads, 0, s->stream>>>(x, y, z, half_width, d_xyz, d_rgb);
	VRM_CUDA(s, cudaGetLastError());
	rc = vrm_stage_commit(s, total);
	if (rc) return rc;
	if (n_out) *n_out = total;
	return VRM_OK;
}

int vrm_scene_generate_sphere(vrm_scene* s, uint32_t x, uint32_t y, uint32_t z, uint32_t radius, int checkered, uint64_t* n_out)
{
	int rc = check_generate(s);
	if (rc) return rc;
	// the reference's unsigned loop bounds need pos >= radius; its colour ramp divides by 2 * radius and by x + radius - (z - radius)
	if (radius < 2 || radius > 256 || x < radius || y < radius || z < radius || x > (1u << 22) || y > (1u << 22) || z > (1u << 22) || x + radius == z - radius)
	{ s->lastError = "sphere: need 2 <= radius <= 256, every centre coordinate >= radius, x + radius != z - radius"; return VRM_ERR_INVALID; }
	const uint32_t step = checkered ? 2u : 1u;
	const uint64_t n = 2ull * radius, nx = (n + step - 1) / step, candidates = nx * n * n;
	Buf flags, pos;
	VRM_CUDA(s, cudaMalloc(&flags.p, candidates * 4));
	VRM_CUDA(s, cudaMalloc(&pos.p, candidates * 4));
	sphere_flag_kernel<<<grid_for(candidates), kThreads, 0, s->stream>>>(x, y, z, radius, step, candidates, flags.as<uint32_t>());
	uint64_t total = 0;
	rc = scan_counts(s, flags.as<uint32_t>(), pos.as<uint32_t>(), candidates, &total);
	if (rc) return rc;
	if (total == 0) { if (n_out) *n_out = 0; return VRM_OK; }
	int32_t* d_xyz = nullptr; uint32_t* d_rgb = nullptr;
	rc = vrm_stage_reserve(s, total, &d_xyz, &d_rgb);  // appended to the scene's staging arrays, in insertion order
	if (rc) return rc;
sphere_fill_kernel<<<grid_for(candidates), kThreads, 0, s->stream>>>(x, y, z, radius, step, candidates, pos.as<uint32_t>(), d_xyz, d_rgb);
	VRM_CUDA(s, cudaGetLastError());
	rc = vrm_stage_commit(s, total);
	if (rc) return rc;
	if (n_out) *n_out = total;
	return VRM_OK;
}

int vrm_scene_generate_sparse_shells(vrm_scene* s, uint32_t size, uint32_t cell, uint32_t seed, uint32_t fill_pct, uint64_t* n_out)
{
	int rc = check_generate(s);
	if (rc) return rc;
	if (cell < 8 || cell > 256 || size < cell || size % cell != 0 || size / cell > 256) { s->lastError = "sparse_shells: need 8 <= cell <= 256, size a multiple of cell, at most 256 cells per axis"; return VRM_ERR_INVALID; }
	const uint32_t n = size / cell;
	const uint64_t cells = (uint64_t)n * n * n;
	const uint32_t maxRadius = cell / 8 + cell / 4;  // exclusive
	Buf shellCounts, cellCounts, starts;
	VRM_CUDA(s, cudaMalloc(&shellCounts.p, (size_t)maxRadius * 4));
	VRM_CUDA(s, cudaMalloc(&cellCounts.p, cells * 4));
	VRM_CUDA(s, cudaMalloc(&starts.p, cells * 4));
	shell_count_kernel<<<maxRadius, kThreads, 0, s->stream>>>(shellCounts.as<uint32_t>());
	shell_cells_kernel<<<grid_for(cells), kThreads, 0, s->stream>>>(n, cell, seed, fill_pct, shellCounts.as<uint32_t>(), cellCounts.as<uint32_t>());
	uint64_t total = 0;
	rc = scan_counts(s, cellCounts.as<uint32_t>(), starts.as<uint32_t>(), cells, &total);
	if (rc) return rc;
	if (total >= (1ull << 32)) { s->lastError = "sparse_shells has more than 2^32 voxels"; return VRM_ERR_INVALID; }
	if (total == 0) { if (n_out) *n_out = 0; return VRM_OK; }
	int32_t* d_xyz = nullptr; uint32_t* d_rgb = nullptr;
	rc = vrm_stage_reserve(s, total, &d_xyz, &d_rgb);  // appended to the scene's staging arrays, in insertion order
	if (rc) return rc;
shell_fill_kernel<<<(unsigned)cells, kThreads, 0, s->stream>>>(n, cell, seed, fill_pct, starts.as<uint32_t>(), d_xyz, d_rgb);
	VRM_CUDA(s, cudaGetLastError());
	rc = vrm_stage_commit(s, total);
	if (rc) return rc;
	if (n_out) *n_out = total;
	return VRM_OK;
}

}  // extern "C"
