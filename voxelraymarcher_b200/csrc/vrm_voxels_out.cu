// vrm_voxels_out.cu -- the stored voxels of a built scene as a voxel list, box by box, in C order (include/vrm_b200.h, "Voxel lists out").
//
// The work scales with the voxels of the region-table cells the box touches, not with the box's cell count:
//   1. clip the box to the region table; list the non-null region-table cells it touches (one 16-byte entry per region, any order);
//   2. count pass: 64 work units per listed region, one warp per unit --
//        VCS: one (x, y) column of 8 clusters along z; per cluster the box's extent inside it becomes a mask per header word (z-range =
//             byte mask, y-range selects bytes, x-range selects word pairs), ANDed with the 16 occupancy words and popc'd -- behind the
//             region's cluster-exists bits, and without loading a colour;
//        hash table: 1/64 of the region's slots; a used slot counts when its decoded coordinate lies in the box;
//   3. exclusive scan of the unit counts (vrm_exclusive_scan_u32); the total is the one value copied to the host;
//   4. fill pass: the same walk writes (key, colour) pairs at unit start + rank, key = the position in the clipped box with per-axis
//      bit widths, (x-x0) << (by+bz) | (y-y0) << bz | (z-z0): 32 bits when the clipped box has at most 2^32 cells, else 64;
//   5. the builder's stable LSD radix sort on the key (vrm_sort_pairs_u32 / _u64): C order of the box;
//   6. write pass: key -> global coordinate, xyz and rgb.
// The storage layouts are decoded through the helpers of vrm_core.cuh (hash_key_decode, slot_*, vcs_*): the format stays known there.
#include "vrm_internal.h"
#include "../../include/vrm_b200.h"

#include <algorithm>

using namespace vrm;

namespace
{

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr uint32_t kUnitsPerRegion = 64;  // VCS: cluster column (cx, cy) = unit; hash table: slot range unit/64 of the region

// The box clipped to the region table, global coordinates [lo, hi), and the key layout over it
struct ClipBox
{
	int lo[3], hi[3];
	int shY, shX;  // key = (x - lo[0]) << shX | (y - lo[1]) << shY | (z - lo[2])
};

template <class K> __device__ __forceinline__ K box_key(const ClipBox& b, int x, int y, int z)
{
	return ((K)(uint32_t)(x - b.lo[0]) << b.shX) | ((K)(uint32_t)(y - b.lo[1]) << b.shY) | (K)(uint32_t)(z - b.lo[2]);
}

__device__ __forceinline__ uint32_t clamp8(int v) { return (uint32_t)min(max(v, 0), 8); }

// 1. Every non-null region-table cell of the clipped range [u0, u0 + n) (table coordinates): {dense region index, global origin of the
// region}.  Warp-aggregated append; the order is free (the sort orders the list).
__global__ void __launch_bounds__(kThreads) voxels_regions_kernel(SceneView sv, uint32_t u0x, uint32_t u0y, uint32_t u0z, uint32_t nx, uint32_t ny,
                                                                  uint64_t cells, int4* __restrict__ list, uint32_t* __restrict__ nList)
{
	const uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x;
	const uint32_t lane = threadIdx.x & 31u;
	int32_t ri = -1;
	uint32_t ux = 0, uy = 0, uz = 0;
	if (i < cells)
	{
		const uint64_t t = i / nx;  // x fastest, as the table
		ux = u0x + (uint32_t)(i - t * nx);
		uy = u0y + (uint32_t)(t % ny);
		uz = u0z + (uint32_t)(t / ny);
		const uint32_t D = sv.diameter;
		ri = __ldg(sv.regionTable + ((uint64_t)uz * D + uy) * D + ux);
	}
	const uint32_t ball = __ballot_sync(0xFFFFFFFFu, ri >= 0);
	if (!ball) return;
	const int leader = __ffs(ball) - 1;
	uint32_t base = 0;
	if ((int)lane == leader) base = atomicAdd(nList, (uint32_t)__popc(ball));
	base = __shfl_sync(0xFFFFFFFFu, base, leader);
	if (ri >= 0)
		list[base + __popc(ball & ((1u << lane) - 1u))] = make_int4(ri, (sv.minCoord + (int)ux) * kRegion, (sv.minCoord + (int)uy) * kRegion, (sv.minCoord + (int)uz) * kRegion);
}

// 2. / 4. One warp per work unit (grid-stride over the units, so the units of a dense region spread over the warps).
//   !FILL: counts[u] = voxels of unit u inside the box, for u < units (units past the listed regions count 0).
//   FILL:  the unit's voxels as (key, colour) at starts[u] + rank; units with starts[u + 1] == starts[u] are skipped.
template <int ST, bool FILL, class K>
__global__ void __launch_bounds__(kThreads, 4) voxels_units_kernel(SceneView sv, ClipBox b, const int4* __restrict__ list, const uint32_t* __restrict__ nList,
                                                                uint64_t units, uint32_t* __restrict__ counts, K* __restrict__ keys, uint32_t* __restrict__ vals)
{
	const uint32_t lane = threadIdx.x & 31u;
	const uint32_t below = (1u << lane) - 1u;
	const uint64_t nWarps = (uint64_t)gridDim.x * kWarps;
	const uint64_t live = (uint64_t)*nList * kUnitsPerRegion;
	for (uint64_t u = (blockIdx.x * (uint64_t)kThreads + threadIdx.x) >> 5; u < units; u += nWarps)
	{
		uint32_t run = 0;  // FILL: next output position; !FILL: this lane's count
		if (FILL)
		{
			run = counts[u];
			if (counts[u + 1] == run) continue;
		}
		else if (u >= live)
		{
			if (lane == 0) counts[u] = 0u;
			continue;
		}
		const int4 r = list[u / kUnitsPerRegion];  // {ri, global origin x, y, z}
		const uint32_t part = (uint32_t)(u % kUnitsPerRegion);
		if constexpr (ST == kStorageVcs)
		{
			const uint32_t cx = part >> 3, cy = part & 7u;
			const int gx = r.y + 8 * (int)cx, gy = r.z + 8 * (int)cy;
			const uint32_t x0 = clamp8(b.lo[0] - gx), x1 = clamp8(b.hi[0] - gx), y0 = clamp8(b.lo[1] - gy), y1 = clamp8(b.hi[1] - gy);
			if (x0 < x1 && y0 < y1)
			{
				const uint32_t cid0 = vcs_cluster_id(cx, cy, 0u);
				const uint32_t occ = (__ldg(sv.clusterMask + (size_t)r.x * 16 + (cid0 >> 5)) >> (cid0 & 31u)) & 0xFFu;  // clusters cz = 0..7
				const int czLo = max(b.lo[2] - r.w, 0) >> 3, czHi = min((b.hi[2] - r.w + 7) >> 3, 8);
				for (int cz = czLo; cz < czHi; cz++)
				{
					if (!((occ >> cz) & 1u)) continue;
					const int gz = r.w + 8 * cz;
					const uint32_t cid = cid0 | (uint32_t)cz;
					uint2 h = make_uint2(0u, 0u);
					uint32_t m = 0u;
					if (lane < 16u)
					{
						h = __ldg(sv.headers + vcs_header_index((uint32_t)r.x, cid, lane));
						m = h.x & vcs_word_box_mask(lane, x0, x1, y0, y1, clamp8(b.lo[2] - gz), clamp8(b.hi[2] - gz));
					}
					if (!FILL) { run += __popc(m); continue; }
					for (uint32_t w = 0; w < 16u; w++)
					{
						const uint32_t bits = __shfl_sync(0xFFFFFFFFu, m, w);
						if (!bits) continue;
						const uint32_t hx = __shfl_sync(0xFFFFFFFFu, h.x, w), hy = __shfl_sync(0xFFFFFFFFu, h.y, w);
						if ((bits >> lane) & 1u)
						{
							uint32_t x, y, z;
							vcs_word_bit_xyz(w, lane, x, y, z);
							const uint64_t o = run + __popc(bits & below);
							keys[o] = box_key<K>(b, gx + (int)x, gy + (int)y, gz + (int)z);
							vals[o] = __ldg(sv.values + vcs_colour_index(hx, hy, lane));
						}
						run += __popc(bits);
					}
				}
			}
		}
		else
		{
			const RegionRef<kStorageHash> rr = load_region<kStorageHash>(sv, r.x);
			const uint32_t total = 2u * rr.n, len = (total + kUnitsPerRegion - 1u) / kUnitsPerRegion;
			const uint32_t s0 = part * len, s1 = min(s0 + len, total);
			for (uint32_t s = s0; s < s1; s += 32u)
			{
				bool take = false;
				int gx = 0, gy = 0, gz = 0;
				unsigned long long e = kEmptySlot;
				if (s + lane < s1)
				{
					e = __ldg(sv.slots + (rr.base1 + s + lane));
					if (slot_used(e))
					{
						uint32_t x, y, z;
						hash_key_decode(slot_key(e), x, y, z);
						gx = r.y + (int)x; gy = r.z + (int)y; gz = r.w + (int)z;
						take = gx >= b.lo[0] && gx < b.hi[0] && gy >= b.lo[1] && gy < b.hi[1] && gz >= b.lo[2] && gz < b.hi[2];
					}
				}
				if (!FILL) { run += take ? 1u : 0u; continue; }
				const uint32_t ball = __ballot_sync(0xFFFFFFFFu, take);
				if (take)
				{
					const uint64_t o = run + __popc(ball & below);
					keys[o] = box_key<K>(b, gx, gy, gz);
					vals[o] = slot_colour(e);
				}
				run += __popc(ball);
			}
		}
		if (!FILL)
		{
#pragma unroll
			for (int d = 16; d; d >>= 1) run += __shfl_xor_sync(0xFFFFFFFFu, run, d);
			if (lane == 0) counts[u] = run;
		}
	}
}

// 6. sorted keys -> global coordinates
template <class K>
__global__ void __launch_bounds__(kThreads) voxels_write_kernel(const K* __restrict__ keys, const uint32_t* __restrict__ vals, uint64_t n, ClipBox b,
                                                                int32_t* __restrict__ xyz, uint32_t* __restrict__ rgb)
{
	const uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x;
	if (i >= n) return;
	const K k = keys[i];
	xyz[3 * i] = b.lo[0] + (int)(uint32_t)(k >> b.shX);
	xyz[3 * i + 1] = b.lo[1] + (int)((uint32_t)(k >> b.shY) & ((1u << (b.shX - b.shY)) - 1u));
	xyz[3 * i + 2] = b.lo[2] + (int)((uint32_t)k & ((1u << b.shY) - 1u));
	rgb[i] = vals[i];
}

struct Scratch
{
	vrm_scene* s;
	void* p = nullptr;
	explicit Scratch(vrm_scene* sc) : s(sc) {}
	~Scratch() { vrm_free_async(s, p); }
};

size_t pad256(size_t bytes) { return (bytes + 255) & ~size_t(255); }

int bits_for(int64_t extent)
{
	int b = 0;
	while ((int64_t(1) << b) < extent) b++;
	return b;
}

unsigned unit_grid(const vrm_scene* s, uint64_t units)
{
	const uint64_t blocks = (units + kWarps - 1) / kWarps, cap = (uint64_t)s->numSms * 4;  // one resident wave (__launch_bounds__(kThreads, 4))
	return (unsigned)std::max<uint64_t>(1, std::min(blocks, cap));
}

// 4. - 6. for n listed voxels of the units behind `starts` (scanned counts): fill, sort, write into the device outputs
template <class K>
int fill_sort_write(vrm_scene* s, const ClipBox& b, int keyBits, const int4* list, const uint32_t* nList, uint64_t units, uint32_t* starts, uint64_t n,
                    int32_t* d_xyz, uint32_t* d_rgb)
{
	const size_t workElems = vrm_sort_work_elems(n, std::max(keyBits, 1));
	Scratch scratch(s);
	VRM_CUDA(s, vrm_alloc_async(s, &scratch.p, 2 * pad256(n * sizeof(K)) + 2 * pad256(n * 4) + workElems * 4));
	char* c = static_cast<char*>(scratch.p);
	K* keys = reinterpret_cast<K*>(c); c += pad256(n * sizeof(K));
	K* keysB = reinterpret_cast<K*>(c); c += pad256(n * sizeof(K));
	uint32_t* vals = reinterpret_cast<uint32_t*>(c); c += pad256(n * 4);
	uint32_t* valsB = reinterpret_cast<uint32_t*>(c); c += pad256(n * 4);
	uint32_t* work = reinterpret_cast<uint32_t*>(c);
	const SceneView sv = s->view();
	if (s->storage == VRM_STORAGE_HASHTABLE)
		voxels_units_kernel<kStorageHash, true, K><<<unit_grid(s, units), kThreads, 0, s->stream>>>(sv, b, list, nList, units, starts, keys, vals);
	else
		voxels_units_kernel<kStorageVcs, true, K><<<unit_grid(s, units), kThreads, 0, s->stream>>>(sv, b, list, nList, units, starts, keys, vals);
	VRM_CUDA(s, cudaGetLastError());
	if constexpr (sizeof(K) == 4) vrm_sort_pairs_u32(keys, vals, keysB, valsB, n, keyBits, work, s->stream);
	else vrm_sort_pairs_u64(keys, vals, keysB, valsB, n, keyBits, work, s->stream);
	VRM_CUDA(s, cudaGetLastError());
	voxels_write_kernel<K><<<(unsigned)((n + kThreads - 1) / kThreads), kThreads, 0, s->stream>>>(keys, vals, n, b, d_xyz, d_rgb);
	VRM_CUDA(s, cudaGetLastError());
	return VRM_OK;
}

int read_voxels(vrm_scene* s, const int32_t* origin, const uint32_t* dims, int32_t* xyzOut, uint32_t* rgbOut, uint64_t capacity, uint64_t* n_out,
                bool toDevice)
{
	if (n_out) *n_out = 0;
	if (!s || !origin || !dims) return VRM_ERR_INVALID;
	if (!n_out) { s->lastError = "read_voxels: n_out is NULL"; return VRM_ERR_INVALID; }
	if (s->storage < 0) { s->lastError = "scene not built"; return VRM_ERR_STATE; }
	for (int a = 0; a < 3; a++)
		if ((int64_t)origin[a] + (int64_t)dims[a] > (int64_t)INT32_MAX) { s->lastError = "read_voxels: origin + dims overflows int32"; return VRM_ERR_INVALID; }
	if ((xyzOut == nullptr) != (rgbOut == nullptr)) { s->lastError = "read_voxels: exactly one output pointer is NULL"; return VRM_ERR_INVALID; }
	if (toDevice && ((reinterpret_cast<uintptr_t>(xyzOut) | reinterpret_cast<uintptr_t>(rgbOut)) & 3u))
	{ s->lastError = "device outputs must be 4-byte aligned"; return VRM_ERR_INVALID; }
	if (dims[0] == 0 || dims[1] == 0 || dims[2] == 0) return VRM_OK;
	// 1. clip to the region table [64 minCoord, 64 (minCoord + D)) per axis
	ClipBox b;
	uint32_t u0[3], nu[3];
	uint64_t cells = 1;
	const int64_t t0 = (int64_t)kRegion * s->minCoord, t1 = t0 + (int64_t)kRegion * s->diameter;
	for (int a = 0; a < 3; a++)
	{
		const int64_t lo = std::max<int64_t>(origin[a], t0), hi = std::min<int64_t>((int64_t)origin[a] + dims[a], t1);
		if (lo >= hi) return VRM_OK;  // nothing of the box lies in the table
		b.lo[a] = (int)lo; b.hi[a] = (int)hi;
		u0[a] = (uint32_t)((lo >> 6) - s->minCoord);
		nu[a] = (uint32_t)(((hi - 1) >> 6) - s->minCoord) + 1u - u0[a];
		cells *= nu[a];
	}
	const int bx = bits_for(b.hi[0] - b.lo[0]), by = bits_for(b.hi[1] - b.lo[1]), bz = bits_for(b.hi[2] - b.lo[2]);
	b.shY = bz; b.shX = by + bz;
	const int keyBits = bx + by + bz;  // <= 48: at most 65 536 cells per axis (D <= 1024)
	const uint64_t maxRegions = std::min<uint64_t>(s->filled, cells);
	if (maxRegions == 0) return VRM_OK;
	const uint64_t units = maxRegions * kUnitsPerRegion;
	VRM_CUDA(s, cudaSetDevice(s->device));
	// scratch: [list count][region list][unit counts -> starts, units + 1][scan scratch]
	Scratch scratch(s);
	const size_t listBytes = pad256(maxRegions * sizeof(int4)), countBytes = pad256((units + 1) * 4);
	VRM_CUDA(s, vrm_alloc_async(s, &scratch.p, 256 + listBytes + countBytes + vrm_scan_scratch_elems(units + 1) * 4));
	char* c = static_cast<char*>(scratch.p);
	uint32_t* d_nList = reinterpret_cast<uint32_t*>(c);
	int4* d_list = reinterpret_cast<int4*>(c + 256);
	uint32_t* d_counts = reinterpret_cast<uint32_t*>(c + 256 + listBytes);
	uint32_t* d_scan = reinterpret_cast<uint32_t*>(c + 256 + listBytes + countBytes);
	const SceneView sv = s->view();
	VRM_CUDA(s, cudaMemsetAsync(d_nList, 0, 4, s->stream));
	voxels_regions_kernel<<<(unsigned)((cells + kThreads - 1) / kThreads), kThreads, 0, s->stream>>>(sv, u0[0], u0[1], u0[2], nu[0], nu[1], cells, d_list, d_nList);
	VRM_CUDA(s, cudaGetLastError());
	// 2. + 3. counts of units [0, units] (the last one is always 0), scanned in place: starts[units] = total
	if (s->storage == VRM_STORAGE_HASHTABLE)
		voxels_units_kernel<kStorageHash, false, uint32_t><<<unit_grid(s, units + 1), kThreads, 0, s->stream>>>(sv, b, d_list, d_nList, units + 1, d_counts, nullptr, nullptr);
	else
		voxels_units_kernel<kStorageVcs, false, uint32_t><<<unit_grid(s, units + 1), kThreads, 0, s->stream>>>(sv, b, d_list, d_nList, units + 1, d_counts, nullptr, nullptr);
	VRM_CUDA(s, cudaGetLastError());
	vrm_exclusive_scan_u32(d_counts, d_counts, units + 1, d_scan, s->stream);
	uint32_t total = 0;
	VRM_CUDA(s, cudaMemcpyAsync(&total, d_counts + units, 4, cudaMemcpyDeviceToHost, s->stream));
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	*n_out = total;
	if (!xyzOut || total == 0) return VRM_OK;
	if (capacity < total) { s->lastError = "read_voxels: capacity is below the voxel count (n_out holds the count)"; return VRM_ERR_INVALID; }
	int32_t* d_xyz = xyzOut;
	uint32_t* d_rgb = rgbOut;
	Scratch out(s);
	if (!toDevice)
	{
		VRM_CUDA(s, vrm_alloc_async(s, &out.p, pad256((size_t)total * 12) + (size_t)total * 4));
		d_xyz = static_cast<int32_t*>(out.p);
		d_rgb = reinterpret_cast<uint32_t*>(static_cast<char*>(out.p) + pad256((size_t)total * 12));
	}
	// 4. - 6.
	const bool key32 = keyBits <= 32 && b.shX < 32;  // (a 1 x 2^16 x 2^16 box has 32 key bits but no x field to shift into a 32-bit key)
	const int rc = key32 ? fill_sort_write<uint32_t>(s, b, keyBits, d_list, d_nList, units, d_counts, total, d_xyz, d_rgb)
	                             : fill_sort_write<unsigned long long>(s, b, keyBits, d_list, d_nList, units, d_counts, total, d_xyz, d_rgb);
	if (rc) return rc;
	if (!toDevice)
	{
		VRM_CUDA(s, cudaMemcpyAsync(xyzOut, d_xyz, (size_t)total * 12, cudaMemcpyDeviceToHost, s->stream));
		VRM_CUDA(s, cudaMemcpyAsync(rgbOut, d_rgb, (size_t)total * 4, cudaMemcpyDeviceToHost, s->stream));
		VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	}
	return VRM_OK;
}

}  // namespace

extern "C" {

int vrm_scene_read_voxels(vrm_scene* s, const int32_t origin[3], const uint32_t dims[3], int32_t* xyz_out, uint32_t* rgb_out, uint64_t capacity,
                          uint64_t* n_out)
{
	return read_voxels(s, origin, dims, xyz_out, rgb_out, capacity, n_out, false);
}

int vrm_scene_read_voxels_device(vrm_scene* s, const int32_t origin[3], const uint32_t dims[3], int32_t* d_xyz_out, uint32_t* d_rgb_out,
                                 uint64_t capacity, uint64_t* n_out)
{
	return read_voxels(s, origin, dims, d_xyz_out, d_rgb_out, capacity, n_out, true);
}

}  // extern "C"
