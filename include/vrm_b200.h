/* vrm_b200.h -- C ABI of the B200-native voxel raymarcher hot path (libvrm_b200.so).
 *
 * Drop-in boundary for ONE path of lukeduball/VoxelRaymarcher: construction of the two voxel storage
 * structures + primary-ray generation + both traversal algorithms fused with lookup, shadow ray and lighting.
 * Everything behind this header is hand-written CUDA for sm_100a; there is no CPU fallback: every entry point
 * that needs the GPU returns VRM_ERR_CUDA when no device is usable.
 *
 * Reference interfaces replaced (paths relative to /root/reference/VoxelRaymarcher/src):
 *   vrm_scene_add_voxels      <- VoxelSceneCPU::insertVoxel               geometry/VoxelSceneCPU.cuh:16-46
 *   vrm_scene_build           <- VoxelSceneCPU::generateVoxelScene        geometry/VoxelSceneCPU.cuh:49-93
 *                                + CuckooHashTable ctor                   storage/CuckooHashTable.cuh:20-49,97-178
 *                                + VoxelClusterStore ctor                 storage/VoxelClusterStore.cuh:37-85
 *                                + generateVoxelScene<<<1,1>>>            renderer/Renderer.cuh:1066-1086
 *   vrm_scene_info            <- getArrayDiameter/getArraySize/getMinCoord geometry/VoxelSceneCPU.cuh:107-123
 *   vrm_set_lighting          <- setupConstantValues                      main/Main.cu:26-42
 *   vrm_camera_make           <- Camera::Camera                           renderer/camera/Camera.cuh:11-23
 *   vrm_render[_device|_views]<- runRaymarchingKernel + kernels           main/Main.cu:105-163, renderer/Renderer.cuh:1033-1063
 *   vrm_trace_rays[_device]   <- rayMarchVoxelScene[LongestAxis]          renderer/Renderer.cuh:338-434, 917-1010
 *   vrm_lookup                <- StorageStructure::lookupVoxel/doesVoxelSpaceExist  storage/StorageStructure.cuh:12-17
 *
 * Conventions: plain pointers and sizes only; every function returns an int status (VRM_OK = 0); no exceptions
 * cross the boundary; the caller owns every buffer it passes; one handle = one device + one stream; a handle is
 * not thread-safe, distinct handles may be used from distinct threads.  Unless a name ends in _device, pointers
 * are HOST pointers and the call returns after the result is in the caller's buffer.
 */
#ifndef VRM_B200_H
#define VRM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vrm_scene vrm_scene;

enum
{
	VRM_OK = 0,
	VRM_ERR_INVALID = 1, /* bad argument */
	VRM_ERR_CUDA = 2,    /* CUDA runtime error (no device, launch failure, ...); see vrm_last_error */
	VRM_ERR_STATE = 3,   /* call not legal in the handle's state (e.g. render before build) */
	VRM_ERR_NOMEM = 4,   /* device or host allocation failed */
	VRM_ERR_BUILD = 5    /* structure construction did not converge */
};

/* StorageType, geometry/VoxelFunctions.cuh:37 */
enum { VRM_STORAGE_VCS = 0, VRM_STORAGE_HASHTABLE = 1 };
/* rayMarchFunctionID, main/Main.cu:58-68 */
enum { VRM_ALGO_LONGEST_AXIS = 0, VRM_ALGO_ORIGINAL = 1 };

/* Value returned by lookups for "no voxel" (EMPTY_KEY / EMPTY_VAL, geometry/VoxelFunctions.cuh:20-21). */
#define VRM_EMPTY (1u << 30)

/* Camera = the reference's 60-byte struct as 15 floats: origin, lowerLeftCorner, horizontal, vertical, forward
 * (renderer/camera/Camera.cuh:31-36). */
#define VRM_CAMERA_FLOATS 15

const char* vrm_error_string(int status);
/* Text of the last CUDA/runtime error seen by this handle ("" when none). Never NULL. */
const char* vrm_last_error(const vrm_scene* scene);
/* 1 when a CUDA device is usable in this process, else 0. */
int vrm_device_available(void);
/* pickCudaDevice, main/Main.cu:82-94: number of CUDA devices (0 when none) and a device's name. */
int vrm_device_count(void);
int vrm_device_name(int device, char* out, uint64_t capacity);

int vrm_scene_create(int device, vrm_scene** out);
int vrm_scene_destroy(vrm_scene* scene);

/* Use a caller-provided cudaStream_t (passed as void*; 0 is CUDA's legacy default stream) for all later work of this
 * handle, so that a host framework can order and time the kernels with its own events.  vrm_scene_reset_stream goes
 * back to the handle's own non-blocking stream. */
int vrm_scene_set_stream(vrm_scene* scene, void* cuda_stream);
int vrm_scene_reset_stream(vrm_scene* scene);
int vrm_scene_synchronize(vrm_scene* scene);

/* Append voxels in insertion order: xyz = n x 3 int32, rgb = n x uint32 (r<<16|g<<8|b).  Duplicate coordinates:
 * the last one added wins.  Coordinates must satisfy |c| < 2^23.  Legal only before vrm_scene_build.
 * The voxels go into ONE growable device array per scene (geometric growth, no allocation and no synchronisation per call);
 * calls with few voxels are collected in a host block first and copied in blocks of 2^20.  The host variant may reuse its
 * buffers on return.  The device variant enqueues its copy on the handle's stream: the source must stay valid until work
 * ordered after the call on that stream runs (or until vrm_scene_synchronize). */
int vrm_scene_add_voxels(vrm_scene* scene, const int32_t* xyz, const uint32_t* rgb, uint64_t n);
int vrm_scene_add_voxels_device(vrm_scene* scene, const int32_t* d_xyz, const uint32_t* d_rgb, uint64_t n);
/* VoxelSceneCPU::insertVoxel (geometry/VoxelSceneCPU.cuh:16-46), one voxel per call: a vector append on the host (see above),
 * so the reference's insertion loops port as they are. */
int vrm_scene_insert_voxel(vrm_scene* scene, int32_t x, int32_t y, int32_t z, uint32_t rgb);

/* Procedural scenes generated ON THE GPU straight into the staging list (no host copy of the voxels; SURVEY.md 8f-3;
 * the reference's own generators are host loops calling insertVoxel: geometry/VoxelCube.cuh:10-39, VoxelSphere.cuh:10-66).
 * The voxel sets and colours are those of voxelraymarcher_b200/scenes.py terrain() / sparse_shells() -- the synthetic
 * workloads of BASELINE.json configs 3-5.  max_height 0 = size.  n_out (nullable) receives the number of voxels added.
 * Legal only before vrm_scene_build; can be mixed with vrm_scene_add_voxels. */
int vrm_scene_generate_terrain(vrm_scene* scene, uint32_t size, uint32_t seed, uint32_t max_height, uint64_t* n_out);
int vrm_scene_generate_sparse_shells(vrm_scene* scene, uint32_t size, uint32_t cell, uint32_t seed, uint32_t fill_pct, uint64_t* n_out);
/* The reference's own generators on the GPU, voxel for voxel and IN ITS INSERTION ORDER (overlaps: last insert wins):
 * VoxelCube::generateVoxelCube (geometry/VoxelCube.cuh:10-39: z faces red, x faces green, y faces blue) and
 * VoxelSphere::generateVoxelSphere / generateCheckeredVoxelSphere (geometry/VoxelSphere.cuh:10-66, uint32 colour ramp). */
int vrm_scene_generate_cube(vrm_scene* scene, int32_t x, int32_t y, int32_t z, int32_t half_width, uint64_t* n_out);
int vrm_scene_generate_sphere(vrm_scene* scene, uint32_t x, uint32_t y, uint32_t z, uint32_t radius, int checkered, uint64_t* n_out);

/* ---- dense volumes -------------------------------------------------------------------------------------------------------
 * LAYOUT (every dense entry point): a volume of dims = {nx, ny, nz} at origin = {ox, oy, oz} is a C-contiguous uint32 array
 * indexed [x][y][z] -- element (i*ny + j)*nz + k is the voxel at (ox+i, oy+j, oz+k), z fastest; shape (nx, ny, nz) in numpy /
 * torch.  This is the bit order of a VCS cluster word (x%8 << 6 | y%8 << 3 | z%8), so a z-run of 8 cells shares one occupancy word.
 * The reference has no counterpart: the nearest are a loop of VoxelSceneCPU::insertVoxel over the cells
 * (geometry/VoxelSceneCPU.cuh:16-46) and one StorageStructure::lookupVoxel per cell (storage/StorageStructure.cuh:12-17).
 *
 * vrm_scene_add_dense[_device]: every cell whose value is not empty_value is appended to the staging list IN LINEAR-INDEX
 * ORDER, its value as the colour -- exactly what one vrm_scene_add_voxels call with those voxels in that order appends, so
 * last-insert-wins holds across calls of either kind.  Legal only before vrm_scene_build (VRM_ERR_STATE after).  Every cell of
 * the box must satisfy |c| < 2^23 and the scene must stay below 2^32 staged voxels (VRM_ERR_INVALID otherwise).  A zero
 * dimension adds nothing (n_out = 0).  n_out (nullable) receives the number of voxels added.  The compaction runs on the GPU
 * (count pass, scan, fill pass); it synchronises the handle's stream ONCE to learn the count, then enqueues the fill.
 *   host variant: the volume travels through a bounded device buffer in slabs of whole x-planes (256 MiB; one synchronisation
 *                 per slab); the caller may reuse it on return.
 *   device variant: d_volume must be 4-byte aligned (VRM_ERR_INVALID otherwise); the work is enqueued on the handle's stream and
 *                 d_volume must stay valid until work ordered after the call on that stream runs (or vrm_scene_synchronize). */
int vrm_scene_add_dense(vrm_scene* scene, const uint32_t* volume, const uint32_t dims[3], const int32_t origin[3],
                        uint32_t empty_value, uint64_t* n_out);
int vrm_scene_add_dense_device(vrm_scene* scene, const uint32_t* d_volume, const uint32_t dims[3], const int32_t origin[3],
                               uint32_t empty_value, uint64_t* n_out);

/* Build the chosen structure ON THE GPU (radix sort -> last-wins dedupe -> region directory ->
 * VCS cluster tables or cuckoo insertion).  build_ms (nullable) receives the device time.
 * Extent: the cubic region table spans one range of region indices for all three axes and always contains region 0, so
 * max(0, floor(c_max / 64)) - min(0, floor(c_min / 64)) < 1024 must hold, with c_min and c_max taken over every coordinate of every
 * staged voxel (e.g. up to 65535 when no coordinate is negative, down to -65472 when none is above 63) -- stricter than the
 * |c| < 2^23 of vrm_scene_add_voxels.  A wider scene fails with VRM_ERR_INVALID before the staged voxels are touched.
 * A build that returns an error leaves the handle as if it had not been attempted: the same staged scene (possibly already
 * deduplicated), so voxels added later still win and a retry -- e.g. VRM_STORAGE_HASHTABLE after the VCS index widths were
 * exceeded -- builds that scene.  If the staged voxels cannot be restored (an allocation of 12 bytes per voxel fails, or a
 * CUDA error), they are dropped and every later staging call and vrm_scene_build returns VRM_ERR_STATE. */
int vrm_scene_build(vrm_scene* scene, int storage_type, float* build_ms);

/* diameter^3 = size of the cubic region table, min_coord = lowest region index on any axis (both as in the
 * reference), filled = non-empty regions, unique_voxels = voxels after last-wins dedupe, bytes = device bytes
 * held by the built structure.  Any out pointer may be NULL. */
int vrm_scene_info(const vrm_scene* scene, uint32_t* diameter, int32_t* min_coord, uint32_t* filled,
                   uint64_t* unique_voxels, uint64_t* bytes);

/* Defaults = main/Main.cu:26-42: direction unit(1,1,1), colour (1,1,1), position (10,10,-10), point light off,
 * shadows on. */
int vrm_set_lighting(vrm_scene* scene, const float direction[3], const float colour[3], const float position[3],
                     int use_point_light, int use_shadows);

/* Host-side helpers evaluated with the reference's operation order in IEEE fp32 (no contraction). */
int vrm_camera_make(const float origin[3], const float look_at[3], const float up[3], float fov_degrees,
                    float aspect, float out_camera[VRM_CAMERA_FLOATS]);
int vrm_make_unit_vector(const float v[3], float out[3]);

/* Render one frame.  rgb_out = H x W x 3 bytes, row 0 = top (renderer/Renderer.cuh:1024-1031).
 * hits_out (nullable) = H x W x 4 int32: global voxel x,y,z of the first voxel the pixel's primary ray found and
 * a 0/1 flag.  kernel_ms (nullable) = device time of the render kernel alone.
 * ALIGNMENT: hit records are written with 16-byte stores, so every DEVICE hit buffer (d_hits_out of the *_device entry
 * points) must be 16-byte aligned -- VRM_ERR_INVALID otherwise.  Host buffers may have any alignment: a page-locked
 * hits_out / rgb_out that is suitably aligned is written directly by the kernel, anything else goes through the handle's
 * device buffers and a copy. */
int vrm_render(vrm_scene* scene, const float camera[VRM_CAMERA_FLOATS], const float translation[3], uint32_t scale,
               int algorithm, uint32_t width, uint32_t height, uint8_t* rgb_out, int32_t* hits_out, float* kernel_ms);

/* Same with DEVICE output buffers; asynchronous on the handle's stream (no synchronisation, no timing). */
int vrm_render_device(vrm_scene* scene, const float camera[VRM_CAMERA_FLOATS], const float translation[3],
                      uint32_t scale, int algorithm, uint32_t width, uint32_t height, uint8_t* d_rgb_out,
                      int32_t* d_hits_out);

/* A batch of views in ONE launch: cameras = n_views x 15 floats (host); d_rgb_out = n_views x H x W x 3 (device);
 * d_hits_out nullable.  Asynchronous on the handle's stream. */
int vrm_render_views_device(vrm_scene* scene, const float* cameras, uint32_t n_views, const float translation[3],
                            uint32_t scale, int algorithm, uint32_t width, uint32_t height, uint8_t* d_rgb_out,
                            int32_t* d_hits_out);
/* The same with the frames of consecutive views view_stride frame slots apart in the outputs (view v goes to slot v * view_stride):
 * interleaved sharding of a view batch over GPUs -- rank r of N renders views r, r + N, ... with view_stride = N into the shared frame
 * buffer starting at slot r -- balances views of unequal cost better than contiguous blocks. */
int vrm_render_views_device_strided(vrm_scene* scene, const float* cameras, uint32_t n_views, const float translation[3],
                                    uint32_t scale, int algorithm, uint32_t width, uint32_t height, uint8_t* d_rgb_out,
                                    int32_t* d_hits_out, uint32_t view_stride);

/* Streaming multi-view render into HOST frames (n_views x height x width x 3, view-major): the camera orbit of
 * BASELINE.json configs[3] as one call (the reference renders exactly one frame per process, main/Main.cu:105-163).
 * Pinned (cudaHostAlloc / cudaHostRegister'ed) rgb_out: the kernel stores every view straight into it.  Pageable
 * rgb_out: views are rendered in batches into two device buffers in turn and the copy of a finished batch overlaps the
 * rendering of the next (batch size: VRM_VIEW_BATCH_BYTES, default 256 MiB).  total_ms (nullable): device time from the
 * first launch to the last byte on the host. */
int vrm_render_views(vrm_scene* scene, const float* cameras, uint32_t n_views, const float translation[3], uint32_t scale,
                     int algorithm, uint32_t width, uint32_t height, uint8_t* rgb_out, float* total_ms);

/* Arbitrary world rays: rays = n x 6 floats (origin xyz, direction xyz).  colour_out = n x uint32, the value the
 * reference's rayMarchVoxelScene[LongestAxis] returns (0 = background); hits_out nullable as above.  Outputs are in the
 * caller's ray order; the rays themselves are traced in an order chosen for coherence (sorted by origin cell and direction,
 * VRM_TRACE_SORT=0 disables it) -- rays are independent, so results do not depend on it. */
int vrm_trace_rays(vrm_scene* scene, const float* rays, uint64_t n, const float translation[3], uint32_t scale,
                   int algorithm, uint32_t* colour_out, int32_t* hits_out, float* kernel_ms);
int vrm_trace_rays_device(vrm_scene* scene, const float* d_rays, uint64_t n, const float translation[3],
                          uint32_t scale, int algorithm, uint32_t* d_colour_out, int32_t* d_hits_out);

/* ---- multi-GPU exchange over NVLink peer memory ------------------------------------------------------------------
 * The path's only exchange step is the gather of finished frames on one GPU.  Instead of rendering locally and then
 * running a collective, a rank can hand vrm_render_device / vrm_render_views_device a pointer into the GATHERING GPU's
 * memory: the render kernel then stores its frame (coalesced 96-byte row segments) straight through NVLink / NVSwitch
 * while it computes.  These helpers create such a buffer on the gathering rank (cudaMalloc + CUDA IPC handle, 64 bytes,
 * to be sent to the other processes by any means) and map it in the other processes.  One process per GPU.          */
#define VRM_IPC_HANDLE_BYTES 64
int vrm_peer_alloc(int device, uint64_t bytes, void** d_ptr_out, unsigned char handle_out[VRM_IPC_HANDLE_BYTES]);
int vrm_peer_open(int device, const unsigned char handle[VRM_IPC_HANDLE_BYTES], void** d_ptr_out);
int vrm_peer_close(int device, void* d_ptr);   /* for pointers from vrm_peer_open  */
int vrm_peer_free(int device, void* d_ptr);    /* for pointers from vrm_peer_alloc */
/* cudaMemcpy (device to device, synchronous) between raw device pointers, e.g. out of a peer buffer into a framework tensor. */
int vrm_copy_device(int device, void* d_dst, const void* d_src, uint64_t bytes);

/* Completion flags for the one-process-per-GPU form.  After vrm_scene_set_completion_flag every render launch of the handle
 * (vrm_render_device, vrm_render_views_device[_strided]: one launch = one sequence number) is followed, in stream order, by a
 * store of first_value, first_value + 1, ... with release semantics at system scope into *d_flag -- a word in device memory,
 * normally inside the gatherer's peer buffer (vrm_peer_open), so that the gatherer learns that a rank's frames have landed
 * without a collective.  d_flag NULL switches the signal off.  vrm_wait_flags_device enqueues, on a stream of `device`, a
 * one-warp kernel that returns when every word d_flags[i * stride_words], i < n_flags, has reached min_value (compared modulo
 * 2^32) or timeout_ms has passed, in which case it stores 1 into *d_status (device memory, nullable).  Replaces the per-step
 * 4-byte NCCL all-reduce of round 1; the reference has no counterpart (main/Main.cu:158: cudaDeviceSynchronize on one device). */
int vrm_scene_set_completion_flag(vrm_scene* scene, uint32_t* d_flag, uint32_t first_value);
/* The counting form, for views that are claimed dynamically (nobody knows in advance how many launches a rank will make): every
 * render launch is followed by a system-scope atomic add of its number of views to *d_counter; the gatherer waits for the
 * counter to reach the batch size with vrm_wait_flags_device(..., n_flags = 1, min_value = n_views).  NULL switches it off.
 * vrm_claim_next enqueues on `cuda_stream` a one-thread kernel that takes the next unclaimed view index from *d_counter (a word
 * in the gatherer's memory, system-scope atomic add of 1) and writes it to *h_claimed, page-locked host memory of the caller:
 * synchronise the stream, read the index, render that view -- ranks that finish cheap views early simply claim more. */
int vrm_scene_set_completion_counter(vrm_scene* scene, uint32_t* d_counter);
int vrm_claim_next(int device, void* cuda_stream, uint32_t* d_counter, uint32_t* h_claimed);
int vrm_wait_flags_device(int device, void* cuda_stream, const uint32_t* d_flags, uint32_t n_flags, uint32_t stride_words,
                          uint32_t min_value, uint32_t timeout_ms, int* d_status);

/* SURVEY.md 8b `render_views(handles[], cameras[], nviews, ...)`: ONE process driving several devices.  scenes[i] are built
 * handles holding the same voxels, normally one per device (several on one device work too).  The n_views cameras are claimed
 * dynamically -- every handle keeps two single-view launches in flight and takes the next unclaimed view when one finishes --
 * and every frame is stored by its render kernel straight into the gather buffer on scenes[0]'s device (NVLink peer access;
 * without it: local frame + cudaMemcpyPeerAsync).  rgb_out = n_views x H x W x 3 bytes: a device buffer on scenes[0]'s device
 * when out_on_device != 0, else host memory (copied from the gather buffer at the end).  views_per_scene_out (nullable,
 * n_scenes entries) reports how the views were dealt out; total_ms (nullable) is host wall time of the whole call.  Frames
 * are identical to vrm_render of the same camera.  The call returns when every frame is complete. */
int vrm_render_views_sharded(vrm_scene* const* scenes, uint32_t n_scenes, const float* cameras, uint32_t n_views,
                             const float translation[3], uint32_t scale, int algorithm, uint32_t width, uint32_t height,
                             uint8_t* rgb_out, int out_on_device, uint32_t* views_per_scene_out, float* total_ms);

/* The storage seam on GLOBAL voxel coordinates: out[i] = colour or VRM_EMPTY; exists_out[i] (nullable) =
 * doesVoxelSpaceExist (always 1 inside a non-empty region for the hash table; cluster occupancy for the VCS). */
int vrm_lookup(vrm_scene* scene, const int32_t* xyz, uint64_t n, uint32_t* out, uint8_t* exists_out);

/* A box of a BUILT scene as a dense volume (layout: "dense volumes" above): out[cell] = exactly what vrm_lookup returns for the
 * cell's coordinate, the colour or VRM_EMPTY, for both storage types; cells outside the region table or with |c| >= 2^23 read
 * VRM_EMPTY.  Legal only after vrm_scene_build (VRM_ERR_STATE before); origin + dims must not overflow int32 (VRM_ERR_INVALID);
 * a zero dimension writes nothing.  The scene scene_box = origin (64 * min_coord)^3, dims (64 * diameter)^3 (vrm_scene_info)
 * covers every stored voxel.
 *   host variant: synchronous; the box is read in slabs of whole x-planes through a bounded device buffer (256 MiB), so any box
 *                 that fits in host memory works.
 *   device variant: asynchronous on the handle's stream; d_out must be 4-byte aligned (VRM_ERR_INVALID otherwise). */
int vrm_scene_read_box(vrm_scene* scene, const int32_t origin[3], const uint32_t dims[3], uint32_t* out);
int vrm_scene_read_box_device(vrm_scene* scene, const int32_t origin[3], const uint32_t dims[3], uint32_t* d_out);

/* ---- voxel lists out -----------------------------------------------------------------------------------------------------
 * The sparse counterpart of vrm_scene_read_box: every voxel STORED in the built scene whose coordinate lies in the box
 * [origin, origin + dims), each once, as xyz_out (n x 3 int32) and rgb_out (n x uint32) -- the arrays vrm_scene_add_voxels takes.
 * The colour is exactly what vrm_lookup returns for the coordinate (after last-insert-wins dedupe).
 * ORDER: C order of the box, i.e. sorted by increasing (x, y, z), x slowest and z fastest (the layout of the dense entry points), so the
 * list is the non-VRM_EMPTY cells of vrm_scene_read_box(origin, dims) in linear-index order -- whatever the storage type or hash seeds.
 * The one difference: a voxel stored with a colour EQUAL to VRM_EMPTY is listed here (read_box cannot show it).
 * SIZING: n_out is required and always receives the number of voxels in the box.  xyz_out and rgb_out both NULL: count only (VRM_OK);
 * exactly one of them NULL: VRM_ERR_INVALID; capacity < count: VRM_ERR_INVALID, nothing is written and n_out still holds the count, so
 * the caller can size its buffers and call again.  The whole scene is the scene_box of vrm_scene_read_box; its count is unique_voxels.
 * Legal only after vrm_scene_build (VRM_ERR_STATE before); origin + dims must not overflow int32 (VRM_ERR_INVALID); a zero dimension
 * counts 0 (VRM_OK); boxes partly or wholly outside the region table are legal (nothing is stored there).
 * The work scales with the voxels of the region-table cells the box touches, not with its cell count (count pass over the cluster
 * headers / hash slots of those regions, one synchronisation to learn the count, fill pass, radix sort on a key of the position in the
 * box, write pass).  Device scratch, from the stream-ordered pool: 16 bytes per listed voxel (24 when the box, clipped to the region
 * table, has more than 2^32 cells) plus ~1 byte per voxel of sort histograms, and 272 bytes per region for the smaller of the
 * scene's filled regions and the region-table cells the box touches.
 *   host variant: synchronous; the caller may reuse its buffers on return (the list goes through a device buffer of 16 bytes per voxel).
 *   device variant: d_xyz_out and d_rgb_out must be 4-byte aligned (VRM_ERR_INVALID otherwise); the handle's stream is synchronised
 *                 ONCE to learn the count, the rest is enqueued on it: the outputs are ready in stream order. */
int vrm_scene_read_voxels(vrm_scene* scene, const int32_t origin[3], const uint32_t dims[3], int32_t* xyz_out, uint32_t* rgb_out,
                          uint64_t capacity, uint64_t* n_out);
int vrm_scene_read_voxels_device(vrm_scene* scene, const int32_t origin[3], const uint32_t dims[3], int32_t* d_xyz_out, uint32_t* d_rgb_out,
                                 uint64_t capacity, uint64_t* n_out);

/* ---- hit surfaces --------------------------------------------------------------------------------------------------------
 * How far away each hit is and which face the ray entered through, computed from a hit map the render / trace calls wrote (hits_out:
 * global voxel x, y, z and a 0/1 flag per pixel or ray) and the exact ray.  The reference has no such output (it writes RGB8 only).
 * DEFINITION (IEEE fp32, round to nearest, no contraction; one function, vrm_core.cuh hit_surface, serves the kernel and the tests):
 *   ray:   views -- the pixel's ray of the render: image-plane origin P, unit direction D and len = |P - camera origin| (calculateWorldRay);
 *          rays  -- P = rays[6i .. 6i+2], D = rays[6i+3 .. 6i+5].
 *   local origin s_a = (float)scale * (P_a - translation_a), the transform the traversal applies.
 *   For every axis a (x, y, z in that order) with D_a != 0: t_a = ((float)(D_a > 0 ? h_a : h_a + 1) - s_a) / D_a.  t = the largest t_a,
 *   ties to the earlier axis; that axis gives face = 1 + 2a + (D_a < 0).
 *   depth = len + t / (float)scale for views (world distance from the camera origin along the pixel's ray), t / (float)scale for rays
 *   (world ray parameter: P + depth * D is the entry point).
 *   flag 0: depth +inf, face 0.  No axis with D_a != 0 (never a camera ray): depth NaN, face 0.
 *   Not clamped: a ray depth below 0 (a view depth below len) means the origin lies inside the hit voxel, or the traversal's accumulated
 *   rounding reported a voxel the exact ray only grazes.
 * Layouts: views take the hit map as vrm_render[_views]_device writes it, n_views x height x width x 4 int32 (view-major, row 0 = top);
 * depth_out = n_views x height x width float32 and face_out = the same count of uint8 (rays: n each).  depth_out and face_out are each
 * nullable, not both (VRM_ERR_INVALID).  Zero records return VRM_OK and write nothing.  The calls depend only on their arguments -- the
 * handle lends its device, stream and scratch buffers -- and are legal before and after vrm_scene_build.
 *   host variants: synchronous; hits, rays and outputs travel through the handle's device buffers.
 *   device variants: asynchronous on the handle's stream; d_hits must be 16-byte aligned, d_depth_out and d_rays 4-byte aligned
 *                    (VRM_ERR_INVALID otherwise); cameras stay a HOST array of n_views x 15 floats.
 * Cost: one streaming pass, 16 bytes read and 5 written per record (DESIGN.md §3.6). */
/* face codes: 0 = no hit, 1..6 = -x, +x, -y, +y, -z, +z (outward normal of the entered face) */
int vrm_hit_surface_views(vrm_scene* scene, const float* cameras, uint32_t n_views, const float translation[3], uint32_t scale,
                          uint32_t width, uint32_t height, const int32_t* hits, float* depth_out, uint8_t* face_out);
int vrm_hit_surface_views_device(vrm_scene* scene, const float* cameras, uint32_t n_views, const float translation[3], uint32_t scale,
                                 uint32_t width, uint32_t height, const int32_t* d_hits, float* d_depth_out, uint8_t* d_face_out);
int vrm_hit_surface_rays(vrm_scene* scene, const float* rays, uint64_t n, const float translation[3], uint32_t scale,
                         const int32_t* hits, float* depth_out, uint8_t* face_out);
int vrm_hit_surface_rays_device(vrm_scene* scene, const float* d_rays, uint64_t n, const float translation[3], uint32_t scale,
                                const int32_t* d_hits, float* d_depth_out, uint8_t* d_face_out);

/* ---- exact ray casts -----------------------------------------------------------------------------------------------------
 * The first STORED voxel (one vrm_scene_read_voxels lists) along the exact ray within a ray interval, with its entry depth, face and colour.
 * Unlike vrm_trace_rays / vrm_render, which reproduce the reference's walks and their fp32 drift and always run to the first hit or out of
 * the scene, the result is a pure function of the ray, and the walk ends at t_far.
 * DEFINITION (IEEE fp32, round to nearest, no contraction; one function, vrm_core.cuh cast_ray, serves the kernel and the tests):
 *   local frame: s_a = (float)scale * (P_a - translation_a) for the world origin P and direction D (any length); voxel c occupies
 *     [c_a, c_a + 1) on each axis; the local parameter tau relates to the world ray parameter t by t = tau / scale, and the walk covers
 *     tau0 = t_near * scale .. tau1 = t_far * scale.
 *   plane crossings: for an axis with D_a != 0 (-0.0 counts as zero), plane k is crossed at tau_a(k) = ((float)k - s_a) / D_a -- the
 *     expression of the hit surfaces; monotone in k, not strictly once |k - s_a| passes about 2^23.
 *   start cell: the cell after every crossing with tau <= tau0: c_a = max{k : tau_a(k) <= tau0} for D_a > 0, min{k : tau_a(k + 1) <= tau0}
 *     for D_a < 0, floorf(s_a) for D_a == 0 (a search on tau_a, not floor(s + tau0 * D), which rounds differently).
 *   walk: repeatedly take the smallest next crossing, tau_a(c_a + 1) for D_a > 0 or tau_a(c_a) for D_a < 0, ties to the earlier axis
 *     (x, y, z); stop when it is > tau1, else step c_a by +-1: the new cell was entered at that tau through face 1 + 2a + (D_a < 0).
 *   result: the first cell of that sequence, the start cell included, holding a stored voxel; cells outside the region table's box
 *     [64 * min_coord, 64 * (min_coord + diameter))^3 hold nothing.
 *     hit in an entered cell: hits = {x, y, z, 1}, depth = tau / scale, face 1..6, colour = the stored colour, exactly what vrm_lookup
 *       returns (VRM_EMPTY for a voxel stored with that colour);
 *     hit in the start cell: depth = t_near exactly, face 0;
 *     miss: hits {0, 0, 0, 0}, depth +inf, face 0, colour VRM_EMPTY.
 *   always a miss: a non-finite origin, direction component or t_near, a NaN t_far, t_near > t_far, and a local origin or tau0 that is not
 *     finite in fp32 (a non-finite translation, or an overflow).  A zero direction is legal: only the start cell is tested.
 *   consequences: the depth of an entered-cell hit equals the hit surfaces' depth for that hit record (both take the largest entry-plane
 *     tau), bit for bit except that an exact tie at tau = 0 may give +0 against -0; the face equals theirs except in exact ties between
 *     axes, where the hit surfaces pick the earlier axis and the cast reports the axis it crossed last.  For a scale that is not a power of two, depth can round one ulp outside [t_near, t_far].
 *   views: the pixel's ray of the render (image-plane origin P, unit D, len = |P - camera origin|) over [0, +inf); depth = len + tau / scale,
 *     len for a start-cell hit -- the render's pixel ray traced exactly.  The hit map has the layout vrm_hit_surface_views reads.
 * Layouts: rays = n x 6 floats (origin, direction); ranges = n x 2 floats {t_near, t_far}, NULL = [0, +inf) for every ray; views are
 * view-major n_views x height x width, row 0 = top.  hits_out = records x 4 int32, depth_out float32, face_out uint8 (codes as above),
 * colour_out uint32.  Each output is nullable, not all four (VRM_ERR_INVALID).  Legal only after vrm_scene_build (VRM_ERR_STATE before);
 * scale 0 is VRM_ERR_INVALID; zero records return VRM_OK and write nothing.  Outputs are in the caller's ray order.
 *   host variants: synchronous; rays, ranges and outputs travel through the handle's device buffers.
 *   device variants: asynchronous on the handle's stream; d_hits_out must be 16-byte aligned, d_rays, d_ranges, d_depth_out and
 *                    d_colour_out 4-byte aligned (VRM_ERR_INVALID otherwise); cameras stay a HOST array of n_views x 15 floats.
 * Cost: the walk leaps over null 64^3 regions and empty 8^3 clusters exactly and steps cell by cell only inside occupied clusters
 * (DESIGN.md §3.7). */
int vrm_cast_rays(vrm_scene* scene, const float* rays, const float* ranges, uint64_t n, const float translation[3], uint32_t scale,
                  int32_t* hits_out, float* depth_out, uint8_t* face_out, uint32_t* colour_out);
int vrm_cast_rays_device(vrm_scene* scene, const float* d_rays, const float* d_ranges, uint64_t n, const float translation[3], uint32_t scale,
                         int32_t* d_hits_out, float* d_depth_out, uint8_t* d_face_out, uint32_t* d_colour_out);
int vrm_cast_views(vrm_scene* scene, const float* cameras, uint32_t n_views, const float translation[3], uint32_t scale, uint32_t width,
                   uint32_t height, int32_t* hits_out, float* depth_out, uint8_t* face_out, uint32_t* colour_out);
int vrm_cast_views_device(vrm_scene* scene, const float* cameras, uint32_t n_views, const float translation[3], uint32_t scale, uint32_t width,
                          uint32_t height, int32_t* d_hits_out, float* d_depth_out, uint8_t* d_face_out, uint32_t* d_colour_out);

/* Opt-in L2 residency hint: an access-policy window (persisting) over the structure's hottest array -- the VCS cluster
 * headers or the hash table's slots -- on the handle's current stream (also VRM_L2_PERSIST=1 at vrm_scene_create).  Off by
 * default: on the BASELINE scenes the touched working set already lives in L1/L2 and the window measured no gain. */
int vrm_set_l2_persistence(vrm_scene* scene, int enabled);

/* Event counters of the LAST render / trace call made with statistics enabled (vrm_set_statistics(scene, 1)):
 * out[0] exist checks, [1] exist checks answering false, [2] lookups, [3] lookups that found a voxel,
 * [4] hash table-2 probes, [5] region-table reads, [6] rays, [7] cluster-skip iterations that were fast-forwarded
 * (they are included in [0] and [1]).  Used for the roofline's algorithmic bytes. */
/* enabled: 0 off; 1 counters comparable with the reference's own (every shadow ray traced, as it does); 2 counters of the work as
 * executed by the production kernels, which skip the shadow ray of a pixel that is black already (colour * !shadow = 0). */
int vrm_set_statistics(vrm_scene* scene, int enabled);
int vrm_get_statistics(vrm_scene* scene, uint64_t out[8]);

/* Measurement only (bench.py, tools/l2_bw.py): the device's L2 rates for an L2-resident working set of the given size -- 8-byte
 * random gathers (loads per nanosecond and the algorithmic GB/s they amount to) and a coalesced streaming read.  These are the
 * memory roofs of the traversal kernels, whose working set lives in L2 (SURVEY.md 8d); MEASURED_PEAKS.json only has the HBM copy rate. */
int vrm_microbench_l2(int device, uint64_t working_set_bytes, float* gather8_loads_per_ns, float* gather8_gbs, float* stream_gbs);

#ifdef __cplusplus
}
#endif
#endif /* VRM_B200_H */
