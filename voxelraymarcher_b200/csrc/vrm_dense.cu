// vrm_dense.cu -- dense uint32 volumes in and out of a scene (include/vrm_b200.h, "Dense volumes").
//
// Layout (stated in the header): a volume of dims {nx, ny, nz} at origin {ox, oy, oz} is a C-contiguous uint32 array indexed
// [x][y][z]; element (i*ny + j)*nz + k is the voxel at (ox+i, oy+j, oz+k), z fastest.
//
// In:  the non-empty cells are compacted ON THE GPU into the scene's staging list in linear-index order -- exactly the list one
//      vrm_scene_add_voxels call with those voxels in that order would append (count pass -> exclusive scan -> fill pass).
// Out: one thread per cell, warps along z, through the storage seam of vrm_core.cuh (region_entry / load_region / space_exists /
//      lookup_voxel), as lookup_kernel does -- out[cell] is what vrm_lookup returns for the cell's coordinate.  The storage
//      format stays known in vrm_core.cuh alone.
#include "vrm_internal.h"
#include "../../include/vrm_b200.h"

using namespace vrm;

namespace
{

constexpr int kThreads = 256;
constexpr int kTileIters = 16;                           // cells per thread and tile
constexpr uint64_t kTileCells = (uint64_t)kThreads * kTileIters;  // 4096 consecutive cells per block and tile
constexpr int kWarps = kThreads / 32;
constexpr int32_t kCoordLimit = 1 << 23;                 // |c| < 2^23 for every stored voxel
constexpr uint64_t kSlabBytes = uint64_t(256) << 20;     // host variants: device slab of whole x-planes

// ---- dense -> staging list ---------------------------------------------------------------------------------------------------

// Count pass: non-empty cells per tile (warp ballot + popc), and their 64-bit total (the scan below is 32-bit: the total is
// checked against 2^32 on the host before any index is used).
__global__ void __launch_bounds__(kThreads) dense_count_kernel(const uint32_t* __restrict__ vol, uint64_t n, uint32_t empty,
                                                               uint32_t* __restrict__ tileCounts, unsigned long long* __restrict__ total)
{
	__shared__ uint32_t warpCount[kWarps];
	const uint64_t base = blockIdx.x * kTileCells;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	uint32_t v[kTileIters];
#pragma unroll
	for (int it = 0; it < kTileIters; it++)
	{
		const uint64_t c = base + (uint64_t)it * kThreads + threadIdx.x;
		v[it] = c < n ? __ldg(vol + c) : empty;
	}
	uint32_t cnt = 0;
#pragma unroll
	for (int it = 0; it < kTileIters; it++) cnt += __popc(__ballot_sync(0xFFFFFFFFu, v[it] != empty));
	if (lane == 0) warpCount[warp] = cnt;
	__syncthreads();
	if (threadIdx.x == 0)
	{
		uint32_t t = 0;
#pragma unroll
		for (int w = 0; w < kWarps; w++) t += warpCount[w];
		tileCounts[blockIdx.x] = t;
		if (t) atomicAdd(total, (unsigned long long)t);
	}
}

// Fill pass: re-read the tile, rank every non-empty cell inside the block in linear order -- iteration-major, then warp, then
// lane, which is the cell order -- and write its coordinate and value at tileStart[tile] + rank.  Only the written voxels decode
// their linear index (IDX = uint32_t when the volume has fewer than 2^32 cells: 32-bit divisions).
template <class IDX>
__global__ void __launch_bounds__(kThreads) dense_fill_kernel(const uint32_t* __restrict__ vol, uint64_t n, uint32_t empty, const uint32_t* __restrict__ tileStart,
                                                              uint32_t ny, uint32_t nz, int ox, int oy, int oz,
                                                              int32_t* __restrict__ xyz, uint32_t* __restrict__ rgb)
{
	__shared__ uint32_t offs[kTileIters * kWarps];  // exclusive prefix over (iteration, warp)
	const uint64_t base = blockIdx.x * kTileCells;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	uint32_t v[kTileIters], ball[kTileIters];
#pragma unroll
	for (int it = 0; it < kTileIters; it++)
	{
		const uint64_t c = base + (uint64_t)it * kThreads + threadIdx.x;
		v[it] = c < n ? __ldg(vol + c) : empty;
	}
#pragma unroll
	for (int it = 0; it < kTileIters; it++)
	{
		ball[it] = __ballot_sync(0xFFFFFFFFu, v[it] != empty);
		if (lane == 0) offs[it * kWarps + warp] = __popc(ball[it]);
	}
	__syncthreads();
	if (warp == 0)
	{
		// 128 counts, four per lane, scanned in order
		uint32_t c4[4], sum = 0;
#pragma unroll
		for (int q = 0; q < 4; q++) { c4[q] = offs[lane * 4 + q]; sum += c4[q]; }
		uint32_t incl = sum;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1)
		{
			const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
			if (lane >= d) incl += o;
		}
		uint32_t run = incl - sum;
#pragma unroll
		for (int q = 0; q < 4; q++) { offs[lane * 4 + q] = run; run += c4[q]; }
	}
	__syncthreads();
	const uint64_t start = tileStart[blockIdx.x];
	const uint32_t below = (1u << lane) - 1u;
#pragma unroll
	for (int it = 0; it < kTileIters; it++)
	{
		if (v[it] == empty) continue;
		const uint64_t o = start + offs[it * kWarps + warp] + __popc(ball[it] & below);
		const IDX c = (IDX)(base + (uint64_t)it * kThreads + threadIdx.x);
		const IDX row = c / (IDX)nz, i = row / (IDX)ny;
		const IDX k = c - row * (IDX)nz, j = row - i * (IDX)ny;
		xyz[3 * o] = ox + (int)i; xyz[3 * o + 1] = oy + (int)j; xyz[3 * o + 2] = oz + (int)k;
		rgb[o] = v[it];
	}
}

struct Scratch
{
	vrm_scene* s;
	void* p = nullptr;
	explicit Scratch(vrm_scene* sc) : s(sc) {}
	~Scratch() { vrm_free_async(s, p); }
};

bool box_in_coord_range(const int32_t* origin, const uint32_t* dims)
{
	for (int a = 0; a < 3; a++)
	{
		const int64_t lo = origin[a], hi = (int64_t)origin[a] + (int64_t)dims[a] - 1;
		if (lo <= -kCoordLimit || hi >= kCoordLimit) return false;
	}
	return true;
}

// Compacts one device volume (all cells in [0, n)) into the staging list; *added = voxels appended.  Synchronises the stream
// once, to learn the count.
int compact_volume(vrm_scene* s, const uint32_t* d_vol, const uint32_t dims[3], const int32_t origin[3], uint32_t empty, uint64_t* added)
{
	*added = 0;
	const uint64_t n = (uint64_t)dims[0] * dims[1] * dims[2];
	const uint64_t tiles = (n + kTileCells - 1) / kTileCells;
	const size_t countBytes = (tiles * 4 + 15) & ~(size_t)15;
	Scratch scratch(s);
	VRM_CUDA(s, vrm_alloc_async(s, &scratch.p, 16 + countBytes + vrm_scan_scratch_elems(tiles) * 4));
	unsigned long long* d_total = static_cast<unsigned long long*>(scratch.p);
	uint32_t* d_counts = reinterpret_cast<uint32_t*>(static_cast<char*>(scratch.p) + 16);
	uint32_t* d_scan = reinterpret_cast<uint32_t*>(static_cast<char*>(scratch.p) + 16 + countBytes);
	VRM_CUDA(s, cudaMemsetAsync(d_total, 0, 8, s->stream));
	dense_count_kernel<<<(unsigned)tiles, kThreads, 0, s->stream>>>(d_vol, n, empty, d_counts, d_total);
	VRM_CUDA(s, cudaGetLastError());
	vrm_exclusive_scan_u32(d_counts, d_counts, tiles, d_scan, s->stream);  // tile starts, in place
	unsigned long long total = 0;
	VRM_CUDA(s, cudaMemcpyAsync(&total, d_total, 8, cudaMemcpyDeviceToHost, s->stream));
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	if (total == 0) return VRM_OK;
	if (total >= (1ull << 32)) { s->lastError = "dense volume has 2^32 or more non-empty cells"; return VRM_ERR_INVALID; }
	int32_t* d_xyz = nullptr; uint32_t* d_rgb = nullptr;
	int rc = vrm_stage_reserve(s, total, &d_xyz, &d_rgb);  // appended to the scene's staging arrays, in insertion order
	if (rc) return rc;
	if (n < (1ull << 32))
		dense_fill_kernel<uint32_t><<<(unsigned)tiles, kThreads, 0, s->stream>>>(d_vol, n, empty, d_counts, dims[1], dims[2], origin[0], origin[1], origin[2], d_xyz, d_rgb);
	else
		dense_fill_kernel<uint64_t><<<(unsigned)tiles, kThreads, 0, s->stream>>>(d_vol, n, empty, d_counts, dims[1], dims[2], origin[0], origin[1], origin[2], d_xyz, d_rgb);
	VRM_CUDA(s, cudaGetLastError());
	rc = vrm_stage_commit(s, total);
	if (rc) return rc;
	*added = total;
	return VRM_OK;
}

int add_dense(vrm_scene* s, const uint32_t* volume, const uint32_t* dims, const int32_t* origin, uint32_t empty, uint64_t* n_out, bool fromDevice)
{
	if (n_out) *n_out = 0;
	if (!s || !dims || !origin) return VRM_ERR_INVALID;
	if (int rc = vrm_check_staging(s)) return rc;
	if (dims[0] == 0 || dims[1] == 0 || dims[2] == 0) return VRM_OK;
	if (!volume) { s->lastError = "volume is NULL"; return VRM_ERR_INVALID; }
	if (fromDevice && (reinterpret_cast<uintptr_t>(volume) & 3u)) { s->lastError = "device volume must be 4-byte aligned"; return VRM_ERR_INVALID; }
	if (!box_in_coord_range(origin, dims)) { s->lastError = "dense volume: every cell must satisfy |c| < 2^23"; return VRM_ERR_INVALID; }
	VRM_CUDA(s, cudaSetDevice(s->device));
	if (fromDevice)
	{
		uint64_t added = 0;
		const int rc = compact_volume(s, volume, dims, origin, empty, &added);
		if (rc == VRM_OK && n_out) *n_out = added;
		return rc;
	}
	// host volume: slabs of whole x-planes through one device buffer, appended in order
	const uint64_t plane = (uint64_t)dims[1] * dims[2];
	uint64_t planesPerSlab = kSlabBytes / (plane * 4);
	if (planesPerSlab < 1) planesPerSlab = 1;
	if (planesPerSlab > dims[0]) planesPerSlab = dims[0];
	Scratch slab(s);
	VRM_CUDA(s, vrm_alloc_async(s, &slab.p, planesPerSlab * plane * 4));
	uint64_t sum = 0;
	for (uint64_t i0 = 0; i0 < dims[0]; i0 += planesPerSlab)
	{
		const uint64_t np = dims[0] - i0 < planesPerSlab ? dims[0] - i0 : planesPerSlab;
		VRM_CUDA(s, cudaMemcpyAsync(slab.p, volume + i0 * plane, np * plane * 4, cudaMemcpyHostToDevice, s->stream));
		const uint32_t d[3] = {(uint32_t)np, dims[1], dims[2]};
		const int32_t o[3] = {origin[0] + (int32_t)i0, origin[1], origin[2]};
		uint64_t added = 0;
		int rc = compact_volume(s, static_cast<const uint32_t*>(slab.p), d, o, empty, &added);  // synchronises: the slab may be overwritten next
		if (rc) return rc;
		sum += added;
	}
	if (n_out) *n_out = sum;
	return VRM_OK;
}

// ---- scene -> dense box --------------------------------------------------------------------------------------------------------

// One warp = 32 consecutive cells of one z-row of the box (a "segment"); every warp walks a contiguous range of segments, so the
// row decode (two divisions) happens once per warp and launch.  Per cell: the region-table entry; nothing else in a null region;
// VCS: the cluster-exists bit, then the header word and -- only behind its occupancy bit -- the colour; hash table: the cluster
// filter, then the two probes (lookup_voxel).  Stores are coalesced along z.
template <int ST>
__global__ void __launch_bounds__(kThreads) read_box_kernel(SceneView sv, int ox, int oy, int oz, uint32_t ny, uint32_t nz, uint64_t segments,
                                                            uint64_t segPerWarp, uint32_t* __restrict__ out)
{
	const uint64_t warpId = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
	const uint32_t lane = threadIdx.x & 31u;
	uint64_t seg = warpId * segPerWarp;
	if (seg >= segments) return;
	const uint64_t segEnd = seg + segPerWarp < segments ? seg + segPerWarp : segments;
	const uint32_t segPerRow = (nz + 31u) >> 5;
	uint64_t row = seg / segPerRow;
	uint32_t zs = (uint32_t)(seg - row * segPerRow) << 5;
	uint64_t i = row / ny;
	uint32_t j = (uint32_t)(row - i * ny);
	RayCtx<ST, false> c;
	c.sv = sv;
	c.reset();
	PermIdentity p;
	for (; seg < segEnd; seg++)
	{
		const uint32_t k = zs + lane;
		if (k < nz)
		{
			const int v[3] = {ox + (int)i, oy + (int)j, oz + (int)k};
			uint32_t res = kEmpty;
			if (v[0] > -kCoordLimit && v[0] < kCoordLimit && v[1] > -kCoordLimit && v[1] < kCoordLimit && v[2] > -kCoordLimit && v[2] < kCoordLimit)
			{
				int reg[3] = {v[0] >> 6, v[1] >> 6, v[2] >> 6};   // floor(c / 64), VoxelSceneCPU.cuh:19-21
				const int32_t ri = region_entry(c, p, reg);
				if (ri >= 0)
				{
					const RegionRef<ST> r = load_region<ST>(sv, ri);
					const int l0 = v[0] & 63, l1 = v[1] & 63, l2 = v[2] & 63;
					if (space_exists(c, r, p, l0, l1, l2)) res = lookup_voxel(c, r, p, reg, l0, l1, l2);
				}
			}
			out[(row * nz) + k] = res;
		}
		zs += 32u;
		if (zs >= nz) { zs = 0; row++; if (++j == ny) { j = 0; i++; } }
	}
}

int launch_read_box(vrm_scene* s, const int32_t origin[3], const uint32_t dims[3], uint32_t* d_out)
{
	const uint64_t segments = (uint64_t)dims[0] * dims[1] * ((dims[2] + 31u) >> 5);
	const uint64_t warps = (uint64_t)s->numSms * (2048 / 32);  // one resident wave at full occupancy
	uint64_t segPerWarp = (segments + warps - 1) / warps;
	if (segPerWarp < 1) segPerWarp = 1;
	const uint64_t warpsUsed = (segments + segPerWarp - 1) / segPerWarp;
	const unsigned grid = (unsigned)((warpsUsed + kWarps - 1) / kWarps);
	if (s->storage == VRM_STORAGE_HASHTABLE)
		read_box_kernel<kStorageHash><<<grid, kThreads, 0, s->stream>>>(s->view(), origin[0], origin[1], origin[2], dims[1], dims[2], segments, segPerWarp, d_out);
	else
		read_box_kernel<kStorageVcs><<<grid, kThreads, 0, s->stream>>>(s->view(), origin[0], origin[1], origin[2], dims[1], dims[2], segments, segPerWarp, d_out);
	VRM_CUDA(s, cudaGetLastError());
	return VRM_OK;
}

int read_box(vrm_scene* s, const int32_t* origin, const uint32_t* dims, uint32_t* out, bool toDevice)
{
	if (!s || !origin || !dims) return VRM_ERR_INVALID;
	if (s->storage < 0) { s->lastError = "scene not built"; return VRM_ERR_STATE; }
	for (int a = 0; a < 3; a++)
		if ((int64_t)origin[a] + (int64_t)dims[a] > (int64_t)INT32_MAX) { s->lastError = "read_box: origin + dims overflows int32"; return VRM_ERR_INVALID; }
	if (dims[0] == 0 || dims[1] == 0 || dims[2] == 0) return VRM_OK;
	if (!out) { s->lastError = "output is NULL"; return VRM_ERR_INVALID; }
	if (toDevice && (reinterpret_cast<uintptr_t>(out) & 3u)) { s->lastError = "device output must be 4-byte aligned"; return VRM_ERR_INVALID; }
	const uint64_t plane = (uint64_t)dims[1] * dims[2];
	if (plane > (uint64_t)(1ull << 62) / dims[0]) { s->lastError = "read_box: box too large"; return VRM_ERR_INVALID; }
	VRM_CUDA(s, cudaSetDevice(s->device));
	if (toDevice) return launch_read_box(s, origin, dims, out);
	uint64_t planesPerSlab = kSlabBytes / (plane * 4);
	if (planesPerSlab < 1) planesPerSlab = 1;
	if (planesPerSlab > dims[0]) planesPerSlab = dims[0];
	Scratch slab(s);
	VRM_CUDA(s, vrm_alloc_async(s, &slab.p, planesPerSlab * plane * 4));
	for (uint64_t i0 = 0; i0 < dims[0]; i0 += planesPerSlab)
	{
		const uint64_t np = dims[0] - i0 < planesPerSlab ? dims[0] - i0 : planesPerSlab;
		const int32_t o[3] = {origin[0] + (int32_t)i0, origin[1], origin[2]};
		const uint32_t d[3] = {(uint32_t)np, dims[1], dims[2]};
		int rc = launch_read_box(s, o, d, static_cast<uint32_t*>(slab.p));
		if (rc) return rc;
		VRM_CUDA(s, cudaMemcpyAsync(out + i0 * plane, slab.p, np * plane * 4, cudaMemcpyDeviceToHost, s->stream));
		VRM_CUDA(s, cudaStreamSynchronize(s->stream));  // the slab is reused by the next launch; the caller's memory is complete on return
	}
	return VRM_OK;
}

}  // namespace

extern "C" {

int vrm_scene_add_dense(vrm_scene* s, const uint32_t* volume, const uint32_t dims[3], const int32_t origin[3], uint32_t empty_value, uint64_t* n_out)
{
	return add_dense(s, volume, dims, origin, empty_value, n_out, false);
}

int vrm_scene_add_dense_device(vrm_scene* s, const uint32_t* d_volume, const uint32_t dims[3], const int32_t origin[3], uint32_t empty_value, uint64_t* n_out)
{
	return add_dense(s, d_volume, dims, origin, empty_value, n_out, true);
}

int vrm_scene_read_box(vrm_scene* s, const int32_t origin[3], const uint32_t dims[3], uint32_t* out) { return read_box(s, origin, dims, out, false); }

int vrm_scene_read_box_device(vrm_scene* s, const int32_t origin[3], const uint32_t dims[3], uint32_t* d_out) { return read_box(s, origin, dims, d_out, true); }

}  // extern "C"
