// vrm_build.cu -- voxel staging and GPU construction of the two voxel storage structures (sm_100a).
//
// Replaces the reference's HOST builders (SURVEY.md F4):
//   VoxelSceneCPU::insertVoxel / generateVoxelScene   geometry/VoxelSceneCPU.cuh:16-93   (std::unordered_map per region)
//   CuckooHashTable ctor + createCuckooHashTable      storage/CuckooHashTable.cuh:20-49,97-178 (sequential eviction loop)
//   VoxelClusterStore ctor                            storage/VoxelClusterStore.cuh:37-85 (bucket + std::sort per cluster)
//   generateVoxelScene<<<1,1>>>                       renderer/Renderer.cuh:1066-1086    (serial device-side new)
//
// Staging: voxels arrive in ONE growable pair of device arrays (xyz, rgb) in insertion order; single-voxel inserts are
// collected in a host block first.  The region extent (VoxelSceneCPU.cuh:28-35,129-130) is reduced as the voxels arrive.
//
// Build pipeline (all on the handle's stream; scratch from the device's memory pool, so a second build allocates nothing new):
//   1. key = regionCell << 18 | clusterId << 9 | inClusterCode (cluster-major order).  32 bits when they suffice
//      (region tables up to 2^14 cells, i.e. every scene up to ~1500^3), 64 bits otherwise.  The colours stay where they are.
//   2. stable LSD radix sort, hand-written (histogram / scan / warp-match ranked scatter), digits of up to 9 bits: a 512^3 scene
//      (27 key bits) sorts in 3 passes.  The ping-pong partner buffers are carved out of the xyz staging array, which is dead
//      after step 1 -- the sort allocates only the first key array.
//   3. last-write-wins dedupe (stable sort keeps insertion order inside an equal-key run; keep the run's last).  A scene
//      without duplicates (the usual case) skips the compaction: the sorted arrays ARE the unique arrays.
//   4. region directory: first voxel per occupied table cell, dense region index = rank of the cell among the occupied
//      cells (a scan over the TABLE, not over the voxels); cubic table index ux + uy*D + uz*D*D.
//   5a. VCS: per cluster 16 x {32-bit occupancy mask, index of the word's first colour}; per region a 512-bit
//       cluster-exists mask; colours stay in sorted order, so rank = popcount prefix (no binary search)
//   5b. cuckoo: region descriptors from the region directory on the device (slot bases = a scan over the regions); parallel
//       insertion with 64-bit atomicExch eviction chains into per-region table pairs; regions whose chain bound is hit are
//       cleared and re-inserted with fresh seeds by the next round (CuckooHashTable.cuh:118-129 does the same on the host
//       with a 300 000-eviction bound) -- rounds are launched three at a time and the host looks once per batch.
// Host round trips per build: the region extent, {unique voxels, regions} and (hash table) the convergence flag.
// Only key -> colour (last insert wins) and cluster occupancy are observable through the lookup seam, so the
// layouts are free (SURVEY.md §7 hard part 4).
#include "vrm_internal.h"

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include "../../include/vrm_b200.h"

#include <algorithm>

using namespace vrm;

namespace
{

constexpr int kThreads = 256;
constexpr int kSortItems = 8;                       // keys per thread in the radix passes
constexpr int kSortTile = kThreads * kSortItems;    // 2048 keys per block
constexpr int kMaxDigitBits = 9;
constexpr int kMaxBins = 1 << kMaxDigitBits;
constexpr int kScanItems = 8;
constexpr int kScanTile = kThreads * kScanItems;
constexpr int kMaxEvictions = 400;
constexpr int kMaxRebuilds = 24;
constexpr int kRoundsPerBatch = 3;

// Scratch that lives for one build (stream-ordered: freed when the build's work is done, reused by the next build)
struct PoolBuf
{
	vrm_scene* s = nullptr;
	void* p = nullptr;
	size_t bytes = 0;
	explicit PoolBuf(vrm_scene* scene) : s(scene) {}
	PoolBuf(const PoolBuf&) = delete;
	PoolBuf& operator=(const PoolBuf&) = delete;
	~PoolBuf() { if (p) vrm_free_async(s, p); }
	cudaError_t alloc(size_t n) { bytes = n; return vrm_alloc_async(s, &p, n ? n : 16); }
	template <class T> T* as() { return static_cast<T*>(p); }
	void* release() { void* q = p; p = nullptr; return q; }
};

__host__ __device__ __forceinline__ int floor_div64(int v) { return v >> 6; }  // == floorf(v / 64.0f) for |v| < 2^24 (VoxelSceneCPU.cuh:19-21)

// ---- region extent of newly staged voxels ---------------------------------------------------------------------------
__global__ void region_minmax_kernel(const int32_t* __restrict__ xyz, uint64_t n, int* __restrict__ minmax)
{
	int lo = 0, hi = 0;  // the reference initialises both to 0 (VoxelSceneCPU.cuh:129-130)
	for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n * 3; i += (uint64_t)gridDim.x * blockDim.x)
	{
		int r = floor_div64(xyz[i]);
		lo = min(lo, r); hi = max(hi, r);
	}
	for (int o = 16; o; o >>= 1)
	{
		lo = min(lo, __shfl_xor_sync(0xFFFFFFFFu, lo, o));
		hi = max(hi, __shfl_xor_sync(0xFFFFFFFFu, hi, o));
	}
	if ((threadIdx.x & 31) == 0) { atomicMin(minmax, lo); atomicMax(minmax + 1, hi); }
}

// ---- 1. keys -------------------------------------------------------------------------------------------------------
template <class K>
__global__ void make_keys_kernel(const int32_t* __restrict__ xyz, uint64_t n, int minCoord, uint32_t D, K* __restrict__ keys)
{
	uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (i >= n) return;
	int x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
	int rx = floor_div64(x), ry = floor_div64(y), rz = floor_div64(z);
	uint32_t lx = (uint32_t)(x & 63), ly = (uint32_t)(y & 63), lz = (uint32_t)(z & 63);  // ((c % 64) + 64) % 64, VoxelSceneCPU.cuh:24-26
	K region = ((K)(uint32_t)(rz - minCoord) * D + (uint32_t)(ry - minCoord)) * D + (uint32_t)(rx - minCoord);
	uint32_t cid = ((lx >> 3) << 6) | ((ly >> 3) << 3) | (lz >> 3);  // getVoxelClusterID, VoxelClusterStore.cuh:21-24
	uint32_t code = ((lx & 7) << 6) | ((ly & 7) << 3) | (lz & 7);
	keys[i] = (region << 18) | (K)((cid << 9) | code);
}

// ---- exclusive scan (uint32), recursive three-phase -----------------------------------------------------------------
__global__ void scan_tile_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint64_t n, uint32_t* __restrict__ tileSums)
{
	__shared__ uint32_t warpSums[kThreads / 32];
	uint64_t base = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanItems;
	uint32_t v[kScanItems];
	uint32_t sum = 0;
#pragma unroll
	for (int k = 0; k < kScanItems; k++) { v[k] = base + k < n ? in[base + k] : 0u; sum += v[k]; }
	uint32_t incl = sum;
	int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
	if (lane == 31) warpSums[warp] = incl;
	__syncthreads();
	if (warp == 0)
	{
		uint32_t w = lane < kThreads / 32 ? warpSums[lane] : 0u;
		uint32_t wi = w;
		for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, wi, o); if (lane >= o) wi += t; }
		if (lane < kThreads / 32) warpSums[lane] = wi - w;
		if (lane == kThreads / 32 - 1 && tileSums) tileSums[blockIdx.x] = wi;
	}
	__syncthreads();
	uint32_t run = warpSums[warp] + incl - sum;
#pragma unroll
	for (int k = 0; k < kScanItems; k++) { if (base + k < n) out[base + k] = run; run += v[k]; }
}

__global__ void scan_add_kernel(uint32_t* __restrict__ out, uint64_t n, const uint32_t* __restrict__ tileOffsets)
{
	uint64_t base = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanItems;
	uint32_t add = tileOffsets[blockIdx.x];
#pragma unroll
	for (int k = 0; k < kScanItems; k++) if (base + k < n) out[base + k] += add;
}

size_t scan_scratch_elems(uint64_t n)
{
	size_t total = 0;
	while (n > (uint64_t)kScanTile) { n = (n + kScanTile - 1) / kScanTile; total += n; }
	return total + 1;
}

// out may alias in.  scratch must hold scan_scratch_elems(n) uint32.
void exclusive_scan(const uint32_t* in, uint32_t* out, uint64_t n, uint32_t* scratch, cudaStream_t st)
{
	if (n == 0) return;
	uint64_t tiles = (n + kScanTile - 1) / kScanTile;
	if (tiles == 1) { scan_tile_kernel<<<1, kThreads, 0, st>>>(in, out, n, nullptr); return; }
	scan_tile_kernel<<<(unsigned)tiles, kThreads, 0, st>>>(in, out, n, scratch);
	exclusive_scan(scratch, scratch, tiles, scratch + tiles, st);
	scan_add_kernel<<<(unsigned)tiles, kThreads, 0, st>>>(out, n, scratch);
}

// ---- 2. radix sort -------------------------------------------------------------------------------------------------
template <class K>
__global__ void radix_hist_kernel(const K* __restrict__ keys, uint64_t n, int shift, uint32_t digitMask, uint32_t numTiles, uint32_t* __restrict__ hist)
{
	__shared__ uint32_t h[kMaxBins];
	for (uint32_t b = threadIdx.x; b <= digitMask; b += kThreads) h[b] = 0;
	__syncthreads();
	uint64_t base = (uint64_t)blockIdx.x * kSortTile;
#pragma unroll
	for (int k = 0; k < kSortItems; k++)
	{
		uint64_t i = base + (uint64_t)k * kThreads + threadIdx.x;
		if (i < n) atomicAdd(&h[(uint32_t)(keys[i] >> shift) & digitMask], 1u);
	}
	__syncthreads();
	for (uint32_t b = threadIdx.x; b <= digitMask; b += kThreads) hist[(uint64_t)b * numTiles + blockIdx.x] = h[b];  // digit-major so that one scan orders (digit, tile)
}

// Stable scatter: warp w of a tile owns keys [w*256, w*256+256) of the tile and walks them in rounds of 32 consecutive
// keys, so (warp, round, lane) is the input order.  __match_any_sync groups equal digits inside a round.
template <class K>
__global__ void radix_scatter_kernel(const K* __restrict__ keysIn, const uint32_t* __restrict__ valsIn, uint64_t n, int shift, uint32_t digitMask,
                                     uint32_t numTiles, const uint32_t* __restrict__ histScanned, K* __restrict__ keysOut, uint32_t* __restrict__ valsOut)
{
	__shared__ uint32_t cnt[kThreads / 32][kMaxBins];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint32_t bins = digitMask + 1u;
	for (uint32_t i = threadIdx.x; i < (kThreads / 32) * (uint32_t)kMaxBins; i += kThreads) (&cnt[0][0])[i] = 0;
	__syncthreads();
	const uint64_t warpBase = (uint64_t)blockIdx.x * kSortTile + (uint64_t)warp * (32 * kSortItems);
	K key[kSortItems];
	uint32_t rank[kSortItems];
#pragma unroll
	for (int k = 0; k < kSortItems; k++)
	{
		uint64_t i = warpBase + (uint64_t)k * 32 + lane;
		bool valid = i < n;
		key[k] = valid ? keysIn[i] : (K)0;
		uint32_t d = valid ? ((uint32_t)(key[k] >> shift) & digitMask) : 0xFFFFFFFFu;
		uint32_t peers = __match_any_sync(0xFFFFFFFFu, d);
		int leader = __ffs(peers) - 1;
		uint32_t before = __popc(peers & ((1u << lane) - 1u));
		uint32_t prev = 0;
		if (valid && lane == leader) { prev = cnt[warp][d]; cnt[warp][d] = prev + __popc(peers); }
		prev = __shfl_sync(0xFFFFFFFFu, prev, leader);
		rank[k] = prev + before;
		__syncwarp();
	}
	__syncthreads();
	for (uint32_t d = threadIdx.x; d < bins; d += kThreads)
	{
		// exclusive prefix over the warps of this tile, per digit; add the tile's global offset for the digit
		uint32_t run = histScanned[(uint64_t)d * numTiles + blockIdx.x];
		for (int w = 0; w < kThreads / 32; w++) { uint32_t c = cnt[w][d]; cnt[w][d] = run; run += c; }
	}
	__syncthreads();
#pragma unroll
	for (int k = 0; k < kSortItems; k++)
	{
		uint64_t i = warpBase + (uint64_t)k * 32 + lane;
		if (i < n)
		{
			uint32_t d = (uint32_t)(key[k] >> shift) & digitMask;
			uint32_t dst = cnt[warp][d] + rank[k];
			keysOut[dst] = key[k];
			valsOut[dst] = valsIn[i];
		}
	}
}

// ---- 3. dedupe -----------------------------------------------------------------------------------------------------
template <class K>
__global__ void keep_last_kernel(const K* __restrict__ keys, uint64_t n, uint32_t* __restrict__ keep)
{
	uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (i >= n) return;
	keep[i] = (i + 1 == n || keys[i + 1] != keys[i]) ? 1u : 0u;  // last write wins, VoxelSceneCPU.cuh:45
}

template <class K>
__global__ void compact_kernel(const K* __restrict__ keys, const uint32_t* __restrict__ vals, const uint32_t* __restrict__ keep,
                               const uint32_t* __restrict__ pos, uint64_t n, K* __restrict__ ukeys, uint32_t* __restrict__ uvals)
{
	uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (i >= n || !keep[i]) return;
	ukeys[pos[i]] = keys[i];
	uvals[pos[i]] = vals[i];
}

// ---- 4. region directory -------------------------------------------------------------------------------------------
// The first sorted key of every occupied table cell records where the cell's voxels start in the UNIQUE array: pos[i] = kept
// keys before i, and the first kept key at or after i has the same cell (the last key of a duplicate run is always kept).
template <class K>
__global__ void region_heads_kernel(const K* __restrict__ keys, const uint32_t* __restrict__ pos, uint64_t n, uint32_t* __restrict__ cellFirst, uint32_t* __restrict__ cellOcc)
{
	uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (i >= n) return;
	const uint64_t cell = (uint64_t)(keys[i] >> 18);
	if (i != 0 && (uint64_t)(keys[i - 1] >> 18) == cell) return;
	cellFirst[cell] = pos[i];
	cellOcc[cell] = 1u;
}

// counts[0] = unique voxels, counts[1] = occupied cells
__global__ void counts_kernel(const uint32_t* __restrict__ pos, const uint32_t* __restrict__ keep, uint64_t n,
                              const uint32_t* __restrict__ cellRank, const uint32_t* __restrict__ cellOcc, uint64_t cells, uint32_t* __restrict__ counts)
{
	counts[0] = pos[n - 1] + keep[n - 1];
	counts[1] = cellRank[cells - 1] + cellOcc[cells - 1];
}

// regionTable[cell] = dense region index or -1 (index = ux + uy*D + uz*D*D, VoxelSceneCPU.cuh:61-62; entry, Renderer.cuh:1075);
// regionStart[ri] = first unique voxel of the region, regionStart[numRegions] = unique
__global__ void region_table_kernel(const uint32_t* __restrict__ cellFirst, const uint32_t* __restrict__ cellRank, const uint32_t* __restrict__ cellOcc, uint64_t cells,
                                    uint32_t numRegions, uint32_t unique, int32_t* __restrict__ regionTable, uint32_t* __restrict__ regionStart)
{
	uint64_t c = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (c == 0) regionStart[numRegions] = unique;
	if (c >= cells) return;
	if (cellOcc[c])
	{
		const uint32_t ri = cellRank[c];
		regionTable[c] = (int32_t)ri;
		regionStart[ri] = cellFirst[c];
	}
	else regionTable[c] = -1;  // SURVEY.md F10: the reference forgets to clear its table
}

// ---- 5a. voxel cluster store ---------------------------------------------------------------------------------------
template <class K>
__global__ void vcs_fill_kernel(const K* __restrict__ ukeys, const int32_t* __restrict__ regionTable, uint64_t u,
                                uint2* __restrict__ headers, uint32_t* __restrict__ clusterMask)
{
	uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (j >= u) return;
	K k = ukeys[j];
	// The voxels of one 32-bit occupancy word are contiguous in the sorted array: its first voxel owns the word and
	// gathers the (at most 32) bits itself -- no atomics, no contention on the densely filled words of solid terrain.
	if (j != 0 && (ukeys[j - 1] >> 5) == (k >> 5)) return;
	uint32_t ri = (uint32_t)regionTable[(uint64_t)(k >> 18)];
	uint32_t cid = (uint32_t)(k >> 9) & 511u, code = (uint32_t)k & 511u;
	uint32_t mask = 1u << (code & 31);
	for (uint64_t t = j + 1; t < u && t < j + 32; t++)
	{
		K kt = ukeys[t];
		if ((kt >> 5) != (k >> 5)) break;
		mask |= 1u << ((uint32_t)kt & 31);
	}
	// colours are sorted by (region, cluster, code): rank inside the word = popcount below the bit
	headers[((size_t)ri * 512 + cid) * 16 + (code >> 5)] = make_uint2(mask, (uint32_t)j);
	bool firstOfCluster = j == 0 || (ukeys[j - 1] >> 9) != (k >> 9);
	if (firstOfCluster) atomicOr(clusterMask + (size_t)ri * 16 + (cid >> 5), 1u << (cid & 31));
}

// Every occupancy word of a cluster that holds at least one voxel carries kHeaderClusterExists in its colour index, so that one
// 8-byte header load answers doesClusterExist AND the occupancy test (vrm_flat.cuh voxel_test).  One thread per cluster.
__global__ void vcs_flag_clusters_kernel(uint2* __restrict__ headers, const uint32_t* __restrict__ clusterMask, uint64_t numClusters)
{
	uint64_t c = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (c >= numClusters) return;
	if (!((clusterMask[c >> 5] >> (c & 31)) & 1u)) return;
	uint4* words = reinterpret_cast<uint4*>(headers + c * 16);
	for (int w = 0; w < 8; w++)
	{
		uint4 v = words[w];
		v.y |= kHeaderClusterExists; v.w |= kHeaderClusterExists;
		words[w] = v;
	}
}

// Hash storage: the same 512-bit cluster-occupancy mask per region, used as a NEGATIVE FILTER in front of the two probes
// (vrm_core.cuh lookup_voxel): a voxel of a cluster without voxels cannot be in the table.
template <class K>
__global__ void cluster_mask_kernel(const K* __restrict__ ukeys, const int32_t* __restrict__ regionTable, uint64_t u, uint32_t* __restrict__ clusterMask)
{
	uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (j >= u) return;
	K k = ukeys[j];
	if (j != 0 && (ukeys[j - 1] >> 9) == (k >> 9)) return;  // one thread per (region, cluster): the sorted keys keep a cluster's voxels together
	uint32_t cid = (uint32_t)(k >> 9) & 511u;
	atomicOr(clusterMask + (size_t)(uint32_t)regionTable[(uint64_t)(k >> 18)] * 16 + (cid >> 5), 1u << (cid & 31));
}

// ---- 5b. cuckoo hash table -----------------------------------------------------------------------------------------
__host__ __device__ inline uint32_t seed_for(uint32_t ri, uint32_t attempt, uint32_t which)
{
	uint32_t h = ri * 0x9E3779B1u + attempt * 0x85EBCA77u + which * 0xC2B2AE3Du + 0x27D4EB2Fu;
	h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12; h *= 0x297A2D39u; h ^= h >> 15;
	return h | 1u;  // multiply-shift hashing needs an odd multiplier (vrm_core.cuh hash_slot1/2)
}

// slots per table of a region with cnt voxels: 1.25 N as in the reference (CuckooHashTable.cuh:23), +2 so tiny regions can always place
__host__ __device__ inline uint32_t table_slots(uint32_t cnt) { return cnt + cnt / 4u + 2u; }

__global__ void hash_region_sizes_kernel(const uint32_t* __restrict__ regionStart, uint32_t numRegions, uint32_t* __restrict__ sizes)
{
	uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r < numRegions) sizes[r] = 2u * table_slots(regionStart[r + 1] - regionStart[r]);
}

__global__ void hash_region_desc_kernel(const uint32_t* __restrict__ regionStart, const uint32_t* __restrict__ slotBase, uint32_t numRegions, HashRegionDesc* __restrict__ desc)
{
	uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= numRegions) return;
	HashRegionDesc d;
	d.slotBase = slotBase[r];
	d.n = table_slots(regionStart[r + 1] - regionStart[r]);
	d.seed1 = seed_for(r, 0, 1); d.seed2 = seed_for(r, 0, 2);
	desc[r] = d;
}

__global__ void fill_slots_kernel(unsigned long long* __restrict__ slots, uint64_t n)
{
	for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) slots[i] = kEmptySlot;
}

// failCount[round] = regions whose insertion hit the chain bound in that round.  Round r > 0 re-inserts only the regions the end
// of round r - 1 marked in `retry`, and does nothing at all once a round has ended without failures.
template <class K>
__global__ void cuckoo_insert_kernel(const K* __restrict__ ukeys, const uint32_t* __restrict__ uvals, const int32_t* __restrict__ regionTable, uint64_t u,
                                     const HashRegionDesc* __restrict__ desc, unsigned long long* __restrict__ slots,
                                     const uint32_t* __restrict__ retry, uint32_t* __restrict__ failed, const uint32_t* __restrict__ failCount, uint32_t round)
{
	if (round > 0 && failCount[round - 1] == 0u) return;
	uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (j >= u) return;
	K k = ukeys[j];
	uint32_t ri = (uint32_t)regionTable[(uint64_t)(k >> 18)];
	if (round > 0 && !retry[ri]) return;
	HashRegionDesc d = desc[ri];
	uint32_t cid = (uint32_t)(k >> 9) & 511u, code = (uint32_t)k & 511u;
	uint32_t x = ((cid >> 6) << 3) | (code >> 6), y = (((cid >> 3) & 7u) << 3) | ((code >> 3) & 7u), z = ((cid & 7u) << 3) | (code & 7u);
	unsigned long long entry = ((unsigned long long)vrm::hash_key(x, y, z) << 32) | uvals[j];
	unsigned long long* t1 = slots + d.slotBase;
	unsigned long long* t2 = t1 + d.n;
	int table = 0;
	for (int it = 0; it < kMaxEvictions; it++)
	{
		uint32_t key = (uint32_t)(entry >> 32);
		unsigned long long* slot = table == 0 ? t1 + hash_slot1(key, d.seed1, d.n) : t2 + hash_slot2(key, d.seed2, d.n);
		entry = atomicExch(slot, entry);  // evict whoever lives there (CuckooHashTable.cuh:137-151), atomically
		if (entry == kEmptySlot) return;
		table ^= 1;                       // the evicted entry moves to its other table
	}
	failed[ri] = 1u;  // cycle bound hit: the region is rebuilt with new hash seeds (CuckooHashTable.cuh:118-129)
}

// End of a round, one block per region: a region that failed gets fresh seeds, an empty pair of tables and a retry mark.
__global__ void cuckoo_round_end_kernel(unsigned long long* __restrict__ slots, HashRegionDesc* __restrict__ desc, uint32_t* __restrict__ retry,
                                        uint32_t* __restrict__ failed, uint32_t* __restrict__ failCount, uint32_t round)
{
	if (round > 0 && failCount[round - 1] == 0u) return;  // (failCount[round] stays 0)
	const uint32_t ri = blockIdx.x;
	const bool again = failed[ri] != 0u;
	__syncthreads();
	if (threadIdx.x == 0)
	{
		retry[ri] = again ? 1u : 0u;
		failed[ri] = 0u;
		if (again)
		{
			atomicAdd(failCount + round, 1u);
			desc[ri].seed1 = seed_for(ri, round + 1, 1); desc[ri].seed2 = seed_for(ri, round + 1, 2);
		}
	}
	if (!again) return;
	const HashRegionDesc d = desc[ri];  // slotBase and n never change
	for (uint32_t i = threadIdx.x; i < 2 * d.n; i += blockDim.x) slots[(size_t)d.slotBase + i] = kEmptySlot;
}

unsigned grid_for(uint64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

// ---- a failed build gives its voxels back --------------------------------------------------------------------------
// Inverse of make_keys_kernel: the voxel of a key of the region table (D, minCoord).
template <class K>
__global__ void key_to_xyz_kernel(const K* __restrict__ keys, uint64_t n, int minCoord, uint32_t D, int32_t* __restrict__ xyz)
{
	uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if (i >= n) return;
	const K k = keys[i];
	const uint64_t region = (uint64_t)(k >> 18);
	const int rx = (int)(region % D) + minCoord, ry = (int)(region / D % D) + minCoord, rz = (int)(region / D / D) + minCoord;
	const uint32_t cid = (uint32_t)(k >> 9) & 511u, code = (uint32_t)k & 511u;
	xyz[3 * i] = rx * 64 + (int)(((cid >> 6) << 3) | (code >> 6));
	xyz[3 * i + 1] = ry * 64 + (int)((((cid >> 3) & 7u) << 3) | ((code >> 3) & 7u));
	xyz[3 * i + 2] = rz * 64 + (int)(((cid & 7u) << 3) | (code & 7u));
}

// After the sort the staging list is gone: the colours were sorted in place of d_stageRgb and, with 32-bit keys, the sort's partner
// buffers were carved out of d_stageXyz.  A build that fails after that point puts n sorted pairs back as the staged list -- the
// stable-sorted ones (their order keeps last-insert-wins) or the deduplicated ones -- so that the handle stages the same scene as
// before the build.  The keys may live inside d_stageXyz, so they are decoded into a fresh array.  If even that fails, the staging
// is marked lost: later staging and build calls return VRM_ERR_STATE instead of building another scene.
template <class K>
void restage(vrm_scene* s, const K* keys, const uint32_t* vals, uint64_t n, int minCoord, uint32_t D)
{
	int32_t* xyz = nullptr;
	cudaError_t e = vrm_alloc_async(s, reinterpret_cast<void**>(&xyz), n * 12);
	if (e == cudaSuccess)
	{
		key_to_xyz_kernel<K><<<grid_for(n), kThreads, 0, s->stream>>>(keys, n, minCoord, D, xyz);
		e = cudaGetLastError();
	}
	if (e == cudaSuccess && vals != s->d_stageRgb) e = cudaMemcpyAsync(s->d_stageRgb, vals, n * 4, cudaMemcpyDeviceToDevice, s->stream);
	if (e != cudaSuccess)
	{
		cudaGetLastError();
		vrm_free_async(s, xyz);
		vrm_stage_free(s);
		s->nStaged = 0;
		s->stageLost = true;
		s->lastError += " (the staged voxels could not be restored)";
		return;
	}
	vrm_free_async(s, s->d_stageXyz);
	s->d_stageXyz = xyz;
	s->stageCap = n;  // d_stageRgb holds at least n
	s->nStaged = n;
}

// Armed (keys set) once the sort has consumed the staging list; a return while armed hands the pairs back.  Declared after the
// buffers that hold them, so it runs before their stream-ordered frees.
template <class K>
struct RestageOnFailure
{
	vrm_scene* s; int minCoord; uint32_t D;
	const K* keys = nullptr; const uint32_t* vals = nullptr; uint64_t n = 0;
	void arm(const K* k, const uint32_t* v, uint64_t count) { keys = k; vals = v; n = count; }
	~RestageOnFailure() { if (keys) restage(s, keys, vals, n, minCoord, D); }
};

// VRM_BUILD_TRACE=1: host-clock stage marks on stderr (each mark synchronises the stream, so traced builds are slower)
struct BuildTrace
{
	bool on = getenv("VRM_BUILD_TRACE") != nullptr;
	std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
	void mark(cudaStream_t st, const char* what)
	{
		if (!on) return;
		cudaStreamSynchronize(st);
		auto t1 = std::chrono::steady_clock::now();
		fprintf(stderr, "[vrm build] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
		t0 = t1;
	}
};

size_t pad256(size_t bytes) { return (bytes + 255) & ~size_t(255); }

// Everything of the build that depends on the key width.
template <class K>
int build_typed(vrm_scene* s, int storageType, int keyBits, int minCoord, uint64_t D, BuildTrace& trace)
{
	cudaStream_t st = s->stream;
	const uint64_t n = s->nStaged;
	const uint64_t tableSize = D * D * D;

	PoolBuf regionTable(s);
	if (regionTable.alloc(tableSize * sizeof(int32_t)) != cudaSuccess) { cudaGetLastError(); s->lastError = "region table allocation failed"; return VRM_ERR_NOMEM; }

	uint64_t unique = 0;
	uint32_t numRegions = 0;
	PoolBuf keysA(s), extra(s), uniq(s), regionStart(s), cellBuf(s);
	RestageOnFailure<K> restore{s, minCoord, (uint32_t)D};
	K* ukeys = nullptr;
	uint32_t* uvals = nullptr;
	bool valsAreStageRgb = false;  // uvals == s->d_stageRgb: the colour array can change owner without a copy
	if (n == 0) VRM_CUDA(s, cudaMemsetAsync(regionTable.p, 0xFF, tableSize * sizeof(int32_t), st));
	else
	{
		// ---- 1. keys; the colours are sorted in place of the staging array --------------------------------------------
		const uint32_t numTiles = (uint32_t)((n + kSortTile - 1) / kSortTile);
		const int passes = (keyBits + kMaxDigitBits - 1) / kMaxDigitBits;
		const int digitBits = (keyBits + passes - 1) / passes;
		const uint32_t digitMask = (1u << digitBits) - 1u;
		const uint64_t histElems = (uint64_t)(digitMask + 1u) * numTiles;
		const size_t scratchElems = scan_scratch_elems(std::max<uint64_t>(std::max<uint64_t>(histElems, n), tableSize));
		if (keysA.alloc(n * sizeof(K)) != cudaSuccess) { cudaGetLastError(); s->lastError = "build scratch allocation failed"; return VRM_ERR_NOMEM; }
		make_keys_kernel<K><<<grid_for(n), kThreads, 0, st>>>(s->d_stageXyz, n, minCoord, (uint32_t)D, keysA.as<K>());
		// The xyz staging array (12 bytes per voxel) is dead now: the sort's partner buffers, the histograms and the scan scratch are
		// carved out of it when they fit (32-bit keys: 8 bytes per voxel + ~5 %), else out of one extra allocation.
		const size_t needB = pad256(n * sizeof(K)) + pad256(n * 4) + pad256(histElems * 4) + pad256(scratchElems * 4);
		char* carve = reinterpret_cast<char*>(s->d_stageXyz);
		if (needB > (size_t)s->stageCap * 12)
		{
			if (extra.alloc(needB) != cudaSuccess) { cudaGetLastError(); s->lastError = "build scratch allocation failed"; return VRM_ERR_NOMEM; }
			carve = extra.as<char>();
		}
		K* keysB = reinterpret_cast<K*>(carve); carve += pad256(n * sizeof(K));
		uint32_t* valsB = reinterpret_cast<uint32_t*>(carve); carve += pad256(n * 4);
		uint32_t* hist = reinterpret_cast<uint32_t*>(carve); carve += pad256(histElems * 4);
		uint32_t* scratch = reinterpret_cast<uint32_t*>(carve);
		trace.mark(st, "keys");
		// ---- 2. stable LSD radix sort -----------------------------------------------------------------------------------
		K* kin = keysA.as<K>(); K* kout = keysB;
		uint32_t* vin = s->d_stageRgb; uint32_t* vout = valsB;
		for (int p = 0; p < passes; p++)
		{
			const int shift = p * digitBits;
			radix_hist_kernel<K><<<numTiles, kThreads, 0, st>>>(kin, n, shift, digitMask, numTiles, hist);
			exclusive_scan(hist, hist, histElems, scratch, st);
			radix_scatter_kernel<K><<<numTiles, kThreads, 0, st>>>(kin, vin, n, shift, digitMask, numTiles, hist, kout, vout);
			std::swap(kin, kout); std::swap(vin, vout);
		}
		restore.arm(kin, vin, n);
		trace.mark(st, "radix sort");
		// ---- 3. + 4. dedupe flags, region heads, one read-back of {unique, regions} (kout / vout are free now) ------------
		uint32_t* keep = vout;
		uint32_t* pos = reinterpret_cast<uint32_t*>(kout);
		if (cellBuf.alloc(pad256(tableSize * 4) * 3 + 256) != cudaSuccess) { cudaGetLastError(); s->lastError = "region directory allocation failed"; return VRM_ERR_NOMEM; }
		uint32_t* cellFirst = cellBuf.as<uint32_t>();
		uint32_t* cellOcc = reinterpret_cast<uint32_t*>(cellBuf.as<char>() + pad256(tableSize * 4));
		uint32_t* cellRank = reinterpret_cast<uint32_t*>(cellBuf.as<char>() + 2 * pad256(tableSize * 4));
		uint32_t* counts = reinterpret_cast<uint32_t*>(cellBuf.as<char>() + 3 * pad256(tableSize * 4));
		VRM_CUDA(s, cudaMemsetAsync(cellOcc, 0, tableSize * 4, st));
		keep_last_kernel<K><<<grid_for(n), kThreads, 0, st>>>(kin, n, keep);
		exclusive_scan(keep, pos, n, scratch, st);
		region_heads_kernel<K><<<grid_for(n), kThreads, 0, st>>>(kin, pos, n, cellFirst, cellOcc);
		exclusive_scan(cellOcc, cellRank, tableSize, scratch, st);
		counts_kernel<<<1, 1, 0, st>>>(pos, keep, n, cellRank, cellOcc, tableSize, counts);
		uint32_t hostCounts[2] = {0, 0};
		VRM_CUDA(s, cudaMemcpyAsync(hostCounts, counts, sizeof(hostCounts), cudaMemcpyDeviceToHost, st));
		VRM_CUDA(s, cudaStreamSynchronize(st));
		unique = hostCounts[0];
		numRegions = hostCounts[1];
		if (unique == n) { ukeys = kin; uvals = vin; valsAreStageRgb = vin == s->d_stageRgb; }
		else
		{
			// duplicates: compact into an exactly sized pair of arrays
			if (uniq.alloc(pad256(unique * sizeof(K)) + unique * 4) != cudaSuccess) { cudaGetLastError(); s->lastError = "unique voxel allocation failed"; return VRM_ERR_NOMEM; }
			ukeys = uniq.as<K>();
			uvals = reinterpret_cast<uint32_t*>(uniq.as<char>() + pad256(unique * sizeof(K)));
			compact_kernel<K><<<grid_for(n), kThreads, 0, st>>>(kin, vin, keep, pos, n, ukeys, uvals);
			restore.arm(ukeys, uvals, unique);
		}
		trace.mark(st, "dedupe + region heads");
		if (regionStart.alloc(((size_t)numRegions + 1) * 4) != cudaSuccess) { cudaGetLastError(); s->lastError = "region directory allocation failed"; return VRM_ERR_NOMEM; }
		region_table_kernel<<<grid_for(tableSize), kThreads, 0, st>>>(cellFirst, cellRank, cellOcc, tableSize, numRegions, (uint32_t)unique, regionTable.as<int32_t>(), regionStart.as<uint32_t>());
		VRM_CUDA(s, cudaGetLastError());
		trace.mark(st, "region directory");
	}

	uint64_t bytes = tableSize * sizeof(int32_t);
	PoolBuf headers(s), clusterMask(s), hashDesc(s), slots(s), values(s);
	if (storageType == VRM_STORAGE_VCS)
	{
		// Zeroed guard space behind both arrays: the reference can test a voxel with a coordinate of exactly 64 (a ray rebased onto the
		// far face of a region; undefined behaviour there, VoxelClusterStore.cuh:93-99 indexes past its 512-entry table).  Both forms of
		// the traversal OR the per-axis terms of the cluster id, so x = 64 together with y = 64 and / or z = 64 gives up to
		// (8 << 6) | (8 << 3) | 8 = 584 -- for the LAST region that reads up to 73 clusters past the end: 80 clusters of guard.
		constexpr size_t kGuardClusters = 80;
		const size_t headerGuard = kGuardClusters * 16 * sizeof(uint2), maskGuard = 128;  // mask: cluster id 584 = word 18 of the last region
		const size_t headerBytes = (size_t)numRegions * 512 * 16 * sizeof(uint2);
		// 31-bit colour indices (the top bit of a header's index word is the cluster-exists flag), 32-bit header word indices (guard included)
		if (unique >= (1ull << 31) || ((uint64_t)numRegions * 512ull + kGuardClusters) * 16ull >= (1ull << 32)) { s->lastError = "scene too large for the VCS index widths"; return VRM_ERR_INVALID; }
		if (headers.alloc(headerBytes + headerGuard) != cudaSuccess || clusterMask.alloc((size_t)numRegions * 16 * 4 + maskGuard) != cudaSuccess)
		{ cudaGetLastError(); s->lastError = "VCS allocation failed"; return VRM_ERR_NOMEM; }
		VRM_CUDA(s, cudaMemsetAsync(headers.p, 0, headerBytes + headerGuard, st));
		VRM_CUDA(s, cudaMemsetAsync(clusterMask.p, 0, (size_t)numRegions * 16 * 4 + maskGuard, st));
		if (unique)
		{
			vcs_fill_kernel<K><<<grid_for(unique), kThreads, 0, st>>>(ukeys, regionTable.as<int32_t>(), unique, headers.as<uint2>(), clusterMask.as<uint32_t>());
			vcs_flag_clusters_kernel<<<grid_for((uint64_t)numRegions * 512), kThreads, 0, st>>>(headers.as<uint2>(), clusterMask.as<uint32_t>(), (uint64_t)numRegions * 512);
		}
		// the colours outlive the build: the staging array itself when the sort ended there (it changes owner once nothing can fail any
		// more, below), else one device copy
		if (!(unique && valsAreStageRgb))
		{
			if (values.alloc(unique * 4) != cudaSuccess) { cudaGetLastError(); s->lastError = "colour array allocation failed"; return VRM_ERR_NOMEM; }
			if (unique) VRM_CUDA(s, cudaMemcpyAsync(values.p, uvals, unique * 4, cudaMemcpyDeviceToDevice, st));
		}
		VRM_CUDA(s, cudaGetLastError());
		bytes += headerBytes + (size_t)numRegions * 64 + unique * 4;
		trace.mark(st, "vcs tables");
	}
	else
	{
		// upper bound of the slot count (exact bases are computed on the device): sum over regions of 2 * (cnt + cnt / 4 + 2)
		const uint64_t totalSlots = 2ull * (unique + unique / 4 + 2ull * numRegions);
		if (totalSlots >= (1ull << 32)) { s->lastError = "hash table needs more than 2^32 slots"; return VRM_ERR_INVALID; }
		PoolBuf ctl(s);
		// control block of the insertion rounds: [slot bases, later retry marks][failed marks][failures per round][scan scratch]
		const size_t regionWords = (size_t)numRegions + 1;
		const size_t wordsBytes = pad256(regionWords * 4), countBytes = pad256((kMaxRebuilds + 1) * 4);
		if (clusterMask.alloc((size_t)numRegions * 16 * 4 + 64) != cudaSuccess || hashDesc.alloc(regionWords * sizeof(HashRegionDesc)) != cudaSuccess ||
		    slots.alloc((totalSlots + 1) * 8) != cudaSuccess || ctl.alloc(2 * wordsBytes + countBytes + scan_scratch_elems(regionWords) * 4) != cudaSuccess)
		{ cudaGetLastError(); s->lastError = "hash table allocation failed"; return VRM_ERR_NOMEM; }
		VRM_CUDA(s, cudaMemsetAsync(clusterMask.p, 0, (size_t)numRegions * 16 * 4 + 64, st));
		if (numRegions)
		{
			uint32_t* sizes = ctl.as<uint32_t>();
			uint32_t* retry = sizes;  // the bases are consumed (hash_region_desc_kernel) before the first round ends
			uint32_t* failed = reinterpret_cast<uint32_t*>(ctl.as<char>() + wordsBytes);
			uint32_t* failCount = reinterpret_cast<uint32_t*>(ctl.as<char>() + 2 * wordsBytes);
			uint32_t* scanScratch = reinterpret_cast<uint32_t*>(ctl.as<char>() + 2 * wordsBytes + countBytes);
			VRM_CUDA(s, cudaMemsetAsync(failed, 0, wordsBytes + countBytes, st));
			cluster_mask_kernel<K><<<grid_for(unique), kThreads, 0, st>>>(ukeys, regionTable.as<int32_t>(), unique, clusterMask.as<uint32_t>());
			hash_region_sizes_kernel<<<grid_for(numRegions), kThreads, 0, st>>>(regionStart.as<uint32_t>(), numRegions, sizes);
			exclusive_scan(sizes, sizes, numRegions, scanScratch, st);
			hash_region_desc_kernel<<<grid_for(numRegions), kThreads, 0, st>>>(regionStart.as<uint32_t>(), sizes, numRegions, hashDesc.as<HashRegionDesc>());
			fill_slots_kernel<<<148 * 8, kThreads, 0, st>>>(slots.as<unsigned long long>(), totalSlots);
			bool converged = false;
			for (uint32_t round = 0; round < (uint32_t)kMaxRebuilds && !converged; )
			{
				const uint32_t batchEnd = std::min<uint32_t>(round + kRoundsPerBatch, kMaxRebuilds);
				for (; round < batchEnd; round++)
				{
					cuckoo_insert_kernel<K><<<grid_for(unique), kThreads, 0, st>>>(ukeys, uvals, regionTable.as<int32_t>(), unique, hashDesc.as<HashRegionDesc>(),
					                                                              slots.as<unsigned long long>(), retry, failed, failCount, round);
					cuckoo_round_end_kernel<<<numRegions, kThreads, 0, st>>>(slots.as<unsigned long long>(), hashDesc.as<HashRegionDesc>(), retry, failed, failCount, round);
				}
				uint32_t hostFail[kMaxRebuilds] = {};
				VRM_CUDA(s, cudaMemcpyAsync(hostFail, failCount, round * 4, cudaMemcpyDeviceToHost, st));
				VRM_CUDA(s, cudaStreamSynchronize(st));
				for (uint32_t r = 0; r < round; r++) if (hostFail[r] == 0u) converged = true;
				if (trace.on) for (uint32_t r = 0; r < round; r++) fprintf(stderr, "[vrm build] cuckoo round %u: %u regions failed\n", r, hostFail[r]);
			}
			if (!converged) { s->lastError = "cuckoo insertion did not converge"; return VRM_ERR_BUILD; }
			VRM_CUDA(s, cudaGetLastError());
		}
		bytes += (size_t)numRegions * sizeof(HashRegionDesc) + totalSlots * 8 + (size_t)numRegions * 64;
		trace.mark(st, "cuckoo insertion");
	}
	VRM_CUDA(s, cudaEventRecord(s->ev1, st));
	VRM_CUDA(s, cudaStreamSynchronize(st));
	VRM_CUDA(s, cudaGetLastError());

	s->d_regionTable = static_cast<int32_t*>(regionTable.release());
	if (storageType == VRM_STORAGE_VCS)
	{
		s->d_headers = static_cast<uint2*>(headers.release());
		s->d_clusterMask = static_cast<uint32_t*>(clusterMask.release());
		if (unique && valsAreStageRgb) { s->d_values = s->d_stageRgb; s->d_stageRgb = nullptr; }
		else s->d_values = static_cast<uint32_t*>(values.release());
	}
	else
	{
		s->d_hashDesc = static_cast<HashRegionDesc*>(hashDesc.release());
		s->d_clusterMask = static_cast<uint32_t*>(clusterMask.release());
		s->d_slots = static_cast<unsigned long long*>(slots.release());
	}
	s->storage = storageType;
	s->diameter = (uint32_t)D;
	s->minCoord = minCoord;
	s->filled = numRegions;
	s->unique = unique;
	s->bytes = bytes;
	restore.keys = nullptr;
	return VRM_OK;
}

}  // namespace

// ---- pooled, stream-ordered allocation ------------------------------------------------------------------------------------
void vrm_configure_pool(int device)
{
	// Freed blocks stay in the pool (no trim at synchronisation points): the scratch of one build is the scratch of the next.
	cudaMemPool_t pool;
	if (cudaDeviceGetDefaultMemPool(&pool, device) != cudaSuccess) { cudaGetLastError(); return; }
	unsigned long long threshold = ~0ull;
	cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
	cudaGetLastError();
}

cudaError_t vrm_alloc_async(vrm_scene* s, void** p, size_t bytes)
{
	*p = nullptr;
	return cudaMallocAsync(p, bytes ? bytes : 16, s->stream);
}

void vrm_free_async(vrm_scene* s, void* p)
{
	if (p && cudaFreeAsync(p, s->stream) != cudaSuccess) cudaGetLastError();
}

// ---- staging -----------------------------------------------------------------------------------------------------------------
void vrm_stage_free(vrm_scene* s)
{
	vrm_free_async(s, s->d_stageXyz); s->d_stageXyz = nullptr;
	vrm_free_async(s, s->d_stageRgb); s->d_stageRgb = nullptr;
	s->stageCap = 0;
	s->pendingXyz.clear(); s->pendingXyz.shrink_to_fit();
	s->pendingRgb.clear(); s->pendingRgb.shrink_to_fit();
}

static int stage_grow(vrm_scene* s, uint64_t need)
{
	if (need <= s->stageCap) return VRM_OK;
	if (need >= (1ull << 32) - (uint64_t)kSortTile) { s->lastError = "too many voxels for 32-bit indices"; return VRM_ERR_INVALID; }
	// geometric growth; the first block is sized exactly, so a scene added in one call wastes nothing
	uint64_t cap = s->stageCap ? std::max<uint64_t>(need, s->stageCap * 2) : need;
	int32_t* nx = nullptr; uint32_t* nr = nullptr;
	cudaError_t e = vrm_alloc_async(s, reinterpret_cast<void**>(&nx), cap * 12);
	if (e == cudaSuccess) e = vrm_alloc_async(s, reinterpret_cast<void**>(&nr), cap * 4);
	if (e == cudaSuccess && s->nStaged) e = cudaMemcpyAsync(nx, s->d_stageXyz, s->nStaged * 12, cudaMemcpyDeviceToDevice, s->stream);
	if (e == cudaSuccess && s->nStaged) e = cudaMemcpyAsync(nr, s->d_stageRgb, s->nStaged * 4, cudaMemcpyDeviceToDevice, s->stream);
	if (e != cudaSuccess) { vrm_free_async(s, nx); vrm_free_async(s, nr); return vrm_fail_cuda(s, e, "voxel staging allocation"); }
	vrm_free_async(s, s->d_stageXyz); vrm_free_async(s, s->d_stageRgb);
	s->d_stageXyz = nx; s->d_stageRgb = nr; s->stageCap = cap;
	return VRM_OK;
}

int vrm_stage_flush_pending(vrm_scene* s)
{
	const uint64_t n = s->pendingRgb.size();
	if (n == 0) return VRM_OK;
	int rc = stage_grow(s, s->nStaged + n);
	if (rc) return rc;
	// pageable source: cudaMemcpyAsync returns once the block has been staged for DMA, so the vectors can be reused at once
	VRM_CUDA(s, cudaMemcpyAsync(s->d_stageXyz + s->nStaged * 3, s->pendingXyz.data(), n * 12, cudaMemcpyHostToDevice, s->stream));
	VRM_CUDA(s, cudaMemcpyAsync(s->d_stageRgb + s->nStaged, s->pendingRgb.data(), n * 4, cudaMemcpyHostToDevice, s->stream));
	s->pendingXyz.clear(); s->pendingRgb.clear();
	return vrm_stage_commit(s, n);
}

int vrm_stage_reserve(vrm_scene* s, uint64_t extra, int32_t** d_xyz, uint32_t** d_rgb)
{
	int rc = vrm_stage_flush_pending(s);  // insertion order: what was inserted before goes first
	if (rc) return rc;
	rc = stage_grow(s, s->nStaged + extra);
	if (rc) return rc;
	*d_xyz = s->d_stageXyz + s->nStaged * 3;
	*d_rgb = s->d_stageRgb + s->nStaged;
	return VRM_OK;
}

int vrm_stage_commit(vrm_scene* s, uint64_t n)
{
	if (n == 0) return VRM_OK;
	if (!s->d_regionMinMax)
	{
		cudaError_t e = vrm_alloc_async(s, reinterpret_cast<void**>(&s->d_regionMinMax), 2 * sizeof(int));
		if (e == cudaSuccess) e = cudaMemsetAsync(s->d_regionMinMax, 0, 2 * sizeof(int), s->stream);  // both start at 0 (VoxelSceneCPU.cuh:129-130)
		if (e != cudaSuccess) return vrm_fail_cuda(s, e, "region extent allocation");
	}
	region_minmax_kernel<<<(unsigned)std::min<uint64_t>((n * 3 + kThreads - 1) / kThreads, 148 * 16), kThreads, 0, s->stream>>>(s->d_stageXyz + s->nStaged * 3, n, s->d_regionMinMax);
	VRM_CUDA(s, cudaGetLastError());
	s->nStaged += n;
	return VRM_OK;
}

void vrm_free_structure(vrm_scene* s)
{
	vrm_free_async(s, s->d_regionTable); s->d_regionTable = nullptr;
	vrm_free_async(s, s->d_hashDesc); s->d_hashDesc = nullptr;
	vrm_free_async(s, s->d_slots); s->d_slots = nullptr;
	vrm_free_async(s, s->d_headers); s->d_headers = nullptr;
	vrm_free_async(s, s->d_clusterMask); s->d_clusterMask = nullptr;
	vrm_free_async(s, s->d_values); s->d_values = nullptr;
	s->storage = -1; s->bytes = 0; s->filled = 0; s->unique = 0;
}

// ---- shadow horizon map (vrm_core.cuh HorizonView) --------------------------------------------------------------------------------
// One thread per (region-table entry, 32-cluster word of its cluster-exists mask), grid-stride: each occupied cluster of the word
// max-es its depth bound into the cells its widened projection covers.
__global__ void horizon_kernel(HorizonView h, int32_t* __restrict__ cells, const int32_t* __restrict__ regionTable, const uint32_t* __restrict__ clusterMask,
                               uint32_t D)
{
	const unsigned long long total = (unsigned long long)D * D * D * 16ull;
	for (unsigned long long t = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; t < total; t += (unsigned long long)gridDim.x * blockDim.x)
	{
		const unsigned long long e = t >> 4;
		const int32_t ri = __ldg(regionTable + e);
		if (ri < 0) continue;
		const uint32_t w = (uint32_t)(t & 15u);
		uint32_t bits = __ldg(clusterMask + (size_t)ri * 16u + w);
		const uint32_t ux = (uint32_t)(e % D), uy = (uint32_t)((e / D) % D), uz = (uint32_t)(e / ((unsigned long long)D * D));
		while (bits)
		{
			const uint32_t cid = w * 32u + (uint32_t)(__ffs(bits) - 1);
			bits &= bits - 1u;
			horizon_splat(h, ux * 8u + (cid >> 6), uy * 8u + ((cid >> 3) & 7u), uz * 8u + (cid & 7u), [&](uint32_t i, int32_t v) { atomicMax(cells + i, v); });
		}
	}
}

int vrm_build_horizon(vrm_scene* s)
{
	s->horizon.cells = nullptr;
	// only the VCS + longest-axis state machine reads the map (vrm_render.cu: fused render and trace kernels)
	if (!s->horizonEnabled || s->storage != VRM_STORAGE_VCS || !s->light.useShadows) return VRM_OK;
	const PermRuntime p = rank_axes(s->light.dir[0], s->light.dir[1], s->light.dir[2]);
	HorizonView h;
	if (!horizon_setup(s->light.dir, s->diameter, (uint32_t)p.a0, h)) return VRM_OK;
	const size_t n = (size_t)h.nu * h.nv;
	if (s->horizonCap < n)
	{
		vrm_free_async(s, s->d_horizon); s->d_horizon = nullptr; s->horizonCap = 0;
		VRM_CUDA(s, vrm_alloc_async(s, reinterpret_cast<void**>(&s->d_horizon), n * sizeof(int32_t)));
		s->horizonCap = n;
	}
	VRM_CUDA(s, cudaMemsetAsync(s->d_horizon, 0x80, n * sizeof(int32_t), s->stream));  // kHorizonEmpty
	const unsigned long long work = (unsigned long long)s->diameter * s->diameter * s->diameter * 16ull;
	const unsigned blocks = (unsigned)std::min<unsigned long long>((work + 255) / 256, (unsigned long long)s->numSms * 32ull);
	horizon_kernel<<<blocks, 256, 0, s->stream>>>(h, s->d_horizon, s->d_regionTable, s->d_clusterMask, s->diameter);
	VRM_CUDA(s, cudaGetLastError());
	h.cells = s->d_horizon;
	s->horizon = h;
	return VRM_OK;
}

int vrm_build_structure(vrm_scene* s, int storageType, float* buildMs)
{
	cudaStream_t st = s->stream;
	BuildTrace trace;
	VRM_CUDA(s, cudaEventRecord(s->ev0, st));
	int rc = vrm_stage_flush_pending(s);
	if (rc) return rc;
	// region extent: reduced while the voxels were staged, read here
	int hostMinMax[2] = {0, 0};
	if (s->d_regionMinMax)
	{
		VRM_CUDA(s, cudaMemcpyAsync(hostMinMax, s->d_regionMinMax, sizeof(hostMinMax), cudaMemcpyDeviceToHost, st));
		VRM_CUDA(s, cudaStreamSynchronize(st));
	}
	trace.mark(st, "extent");
	const int minCoord = hostMinMax[0];
	const uint64_t D = (uint64_t)(hostMinMax[1] - hostMinMax[0] + 1);
	if (D > 1024) { s->lastError = "region table diameter > 1024 (scene spans more than 65536 voxels)"; return VRM_ERR_INVALID; }
	int regionBits = 0;
	while ((1ull << regionBits) < D * D * D) regionBits++;
	const int keyBits = 18 + regionBits;
	rc = keyBits <= 32 ? build_typed<uint32_t>(s, storageType, keyBits, minCoord, D, trace) : build_typed<unsigned long long>(s, storageType, keyBits, minCoord, D, trace);
	if (rc) return rc;
	// the shadow horizon map is part of the build (and of its time)
	rc = vrm_build_horizon(s);
	if (rc) return rc;
	VRM_CUDA(s, cudaEventRecord(s->ev1, st));
	VRM_CUDA(s, cudaStreamSynchronize(st));
	trace.mark(st, "shadow horizon map");
	if (buildMs) VRM_CUDA(s, cudaEventElapsedTime(buildMs, s->ev0, s->ev1));
	return VRM_OK;
}

// exclusive scan for the other translation units (vrm_generate.cu)
size_t vrm_scan_scratch_elems(uint64_t n) { return scan_scratch_elems(n); }
void vrm_exclusive_scan_u32(const uint32_t* in, uint32_t* out, uint64_t n, uint32_t* scratch, cudaStream_t st) { exclusive_scan(in, out, n, scratch, st); }

// The builder's stable LSD radix sort for other callers (vrm_render.cu orders incoherent rays with it, vrm_voxels_out.cu puts voxel lists
// in C order): n (32- or 64-bit key, 32-bit value) pairs, the low keyBits bits of the key.  `work` holds vrm_sort_work_elems(n, keyBits)
// uint32.  On return keys / vals point at the sorted pair (the input pair or the partner pair, depending on the number of passes).
size_t vrm_sort_work_elems(uint64_t n, int keyBits)
{
	const uint32_t numTiles = (uint32_t)((n + kSortTile - 1) / kSortTile);
	const int passes = (keyBits + kMaxDigitBits - 1) / kMaxDigitBits;
	const int digitBits = (keyBits + passes - 1) / passes;
	const uint64_t histElems = ((uint64_t)1 << digitBits) * numTiles;
	return (size_t)(histElems + 64 + scan_scratch_elems(histElems));
}

// Launches the radix_hist_kernel / radix_scatter_kernel instantiations of build_typed<K>; K = uint32_t or unsigned long long.
template <class K>
static void sort_pairs(K*& keys, uint32_t*& vals, K* keysB, uint32_t* valsB, uint64_t n, int keyBits, uint32_t* work, cudaStream_t st)
{
	if (n == 0 || keyBits <= 0) return;
	const uint32_t numTiles = (uint32_t)((n + kSortTile - 1) / kSortTile);
	const int passes = (keyBits + kMaxDigitBits - 1) / kMaxDigitBits;
	const int digitBits = (keyBits + passes - 1) / passes;
	const uint32_t digitMask = (1u << digitBits) - 1u;
	const uint64_t histElems = (uint64_t)(digitMask + 1u) * numTiles;
	uint32_t* hist = work;
	uint32_t* scratch = work + ((histElems + 63) & ~(uint64_t)63);
	K* kin = keys; K* kout = keysB;
	uint32_t* vin = vals; uint32_t* vout = valsB;
	for (int p = 0; p < passes; p++)
	{
		const int shift = p * digitBits;
		radix_hist_kernel<K><<<numTiles, kThreads, 0, st>>>(kin, n, shift, digitMask, numTiles, hist);
		exclusive_scan(hist, hist, histElems, scratch, st);
		radix_scatter_kernel<K><<<numTiles, kThreads, 0, st>>>(kin, vin, n, shift, digitMask, numTiles, hist, kout, vout);
		std::swap(kin, kout); std::swap(vin, vout);
	}
	keys = kin; vals = vin;
}

void vrm_sort_pairs_u32(uint32_t*& keys, uint32_t*& vals, uint32_t* keysB, uint32_t* valsB, uint64_t n, int keyBits, uint32_t* work, cudaStream_t st)
{
	sort_pairs<uint32_t>(keys, vals, keysB, valsB, n, keyBits, work, st);
}

void vrm_sort_pairs_u64(unsigned long long*& keys, uint32_t*& vals, unsigned long long* keysB, uint32_t* valsB, uint64_t n, int keyBits, uint32_t* work,
                        cudaStream_t st)
{
	sort_pairs<unsigned long long>(keys, vals, keysB, valsB, n, keyBits, work, st);
}
