"""Host-side mirror of the reference's interface for the hot path, over the C ABI of ``libvrm_b200.so``
(``include/vrm_b200.h``).  Names follow the reference (VoxelRaymarcher/src):

* ``VoxelScene.insert_voxel / add_voxels``  <- ``VoxelSceneCPU::insertVoxel``            geometry/VoxelSceneCPU.cuh:16-46
* ``VoxelScene.generate_voxel_scene``       <- ``VoxelSceneCPU::generateVoxelScene``     geometry/VoxelSceneCPU.cuh:49-93
* ``VoxelScene.get_array_diameter / get_array_size / get_min_coord``                    geometry/VoxelSceneCPU.cuh:107-123
* ``Camera``                                <- ``Camera::Camera``                        renderer/camera/Camera.cuh:11-23
* ``VoxelScene.setup_constant_values``      <- ``setupConstantValues``                   main/Main.cu:26-42
* ``VoxelScene.run_raymarching_kernel``     <- ``runRaymarchingKernel``                  main/Main.cu:105-163
* ``StorageType`` / algorithm ids                                                       geometry/VoxelFunctions.cuh:37, main/Main.cu:58-68

There is NO CPU fallback: importing works anywhere (so CPU-only tests can check the library's exports), but every
compute entry point raises ``VrmError`` when the CUDA library or a CUDA device is missing.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VRM_B200_LIB") or os.path.join(HERE, "libvrm_b200.so")   # VRM_B200_LIB: an A/B build of the same library (tools/ab_variants.py)

STORAGE_VCS, STORAGE_HASHTABLE = 0, 1          # StorageType {VOXEL_CLUSTER_STORE, HASH_TABLE}
ALGO_LONGEST_AXIS, ALGO_ORIGINAL = 0, 1        # rayMarchFunctionID
STORAGE = {"vcs": STORAGE_VCS, "hashtable": STORAGE_HASHTABLE}
ALGORITHM = {"longestaxis": ALGO_LONGEST_AXIS, "original": ALGO_ORIGINAL}
EMPTY = 1 << 30                                # EMPTY_KEY / EMPTY_VAL

EXPORTS = [
    "vrm_error_string", "vrm_last_error", "vrm_device_available", "vrm_device_count", "vrm_device_name", "vrm_scene_create", "vrm_scene_destroy",
    "vrm_scene_set_stream", "vrm_scene_reset_stream", "vrm_scene_synchronize", "vrm_scene_add_voxels", "vrm_scene_add_voxels_device", "vrm_scene_insert_voxel",
    "vrm_scene_generate_terrain", "vrm_scene_generate_sparse_shells", "vrm_scene_generate_cube", "vrm_scene_generate_sphere",
    "vrm_scene_build", "vrm_scene_info", "vrm_set_lighting", "vrm_camera_make", "vrm_make_unit_vector", "vrm_render",
    "vrm_render_device", "vrm_render_views_device", "vrm_render_views_device_strided", "vrm_render_views", "vrm_trace_rays", "vrm_trace_rays_device", "vrm_lookup",
    "vrm_set_l2_persistence", "vrm_set_statistics", "vrm_get_statistics", "vrm_peer_alloc", "vrm_peer_open", "vrm_peer_close", "vrm_peer_free", "vrm_copy_device", "vrm_microbench_l2",
    "vrm_scene_set_completion_flag", "vrm_scene_set_completion_counter", "vrm_claim_next", "vrm_wait_flags_device", "vrm_render_views_sharded",
    "vrm_scene_add_dense", "vrm_scene_add_dense_device", "vrm_scene_read_box", "vrm_scene_read_box_device",
    "vrm_scene_read_voxels", "vrm_scene_read_voxels_device",
    "vrm_hit_surface_views", "vrm_hit_surface_views_device", "vrm_hit_surface_rays", "vrm_hit_surface_rays_device",
    "vrm_cast_rays", "vrm_cast_rays_device", "vrm_cast_views", "vrm_cast_views_device",
]

# face codes of the hit surfaces -> outward normal of the face the ray entered through (0 = no hit, then -x, +x, -y, +y, -z, +z)
FACE_NORMALS = np.array([[0, 0, 0], [-1, 0, 0], [1, 0, 0], [0, -1, 0], [0, 1, 0], [0, 0, -1], [0, 0, 1]], np.int8)


class VrmError(RuntimeError):
    pass


_lib = None


def load_library():
    """Load libvrm_b200.so (built in-tree by ``__graft_entry__.build()`` / ``make -C voxelraymarcher_b200/csrc``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VrmError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    vp, u64, u32, i32, ci, f32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.c_int, C.c_float
    sig = {
        "vrm_error_string": (C.c_char_p, [ci]),
        "vrm_last_error": (C.c_char_p, [vp]),
        "vrm_device_available": (ci, []),
        "vrm_device_count": (ci, []),
        "vrm_device_name": (ci, [ci, C.c_char_p, u64]),
        "vrm_scene_create": (ci, [ci, C.POINTER(vp)]),
        "vrm_scene_destroy": (ci, [vp]),
        "vrm_scene_set_stream": (ci, [vp, vp]),
        "vrm_scene_reset_stream": (ci, [vp]),
        "vrm_scene_synchronize": (ci, [vp]),
        "vrm_scene_add_voxels": (ci, [vp, vp, vp, u64]),
        "vrm_scene_add_voxels_device": (ci, [vp, vp, vp, u64]),
        "vrm_scene_insert_voxel": (ci, [vp, i32, i32, i32, u32]),
        "vrm_scene_generate_terrain": (ci, [vp, u32, u32, u32, C.POINTER(u64)]),
        "vrm_scene_generate_sparse_shells": (ci, [vp, u32, u32, u32, u32, C.POINTER(u64)]),
        "vrm_scene_generate_cube": (ci, [vp, i32, i32, i32, i32, C.POINTER(u64)]),
        "vrm_scene_generate_sphere": (ci, [vp, u32, u32, u32, u32, ci, C.POINTER(u64)]),
        "vrm_scene_build": (ci, [vp, ci, C.POINTER(f32)]),
        "vrm_scene_info": (ci, [vp, C.POINTER(u32), C.POINTER(i32), C.POINTER(u32), C.POINTER(u64), C.POINTER(u64)]),
        "vrm_set_lighting": (ci, [vp, vp, vp, vp, ci, ci]),
        "vrm_camera_make": (ci, [vp, vp, vp, f32, f32, vp]),
        "vrm_make_unit_vector": (ci, [vp, vp]),
        "vrm_render": (ci, [vp, vp, vp, u32, ci, u32, u32, vp, vp, C.POINTER(f32)]),
        "vrm_render_device": (ci, [vp, vp, vp, u32, ci, u32, u32, vp, vp]),
        "vrm_render_views_device": (ci, [vp, vp, u32, vp, u32, ci, u32, u32, vp, vp]),
        "vrm_render_views_device_strided": (ci, [vp, vp, u32, vp, u32, ci, u32, u32, vp, vp, u32]),
        "vrm_render_views": (ci, [vp, vp, u32, vp, u32, ci, u32, u32, vp, C.POINTER(f32)]),
        "vrm_trace_rays": (ci, [vp, vp, u64, vp, u32, ci, vp, vp, C.POINTER(f32)]),
        "vrm_trace_rays_device": (ci, [vp, vp, u64, vp, u32, ci, vp, vp]),
        "vrm_lookup": (ci, [vp, vp, u64, vp, vp]),
        "vrm_peer_alloc": (ci, [ci, u64, C.POINTER(vp), vp]),
        "vrm_peer_open": (ci, [ci, vp, C.POINTER(vp)]),
        "vrm_peer_close": (ci, [ci, vp]),
        "vrm_peer_free": (ci, [ci, vp]),
        "vrm_copy_device": (ci, [ci, vp, vp, u64]),
        "vrm_set_l2_persistence": (ci, [vp, ci]),
        "vrm_set_statistics": (ci, [vp, ci]),
        "vrm_get_statistics": (ci, [vp, vp]),
        "vrm_microbench_l2": (ci, [ci, u64, C.POINTER(f32), C.POINTER(f32), C.POINTER(f32)]),
        "vrm_scene_set_completion_flag": (ci, [vp, vp, u32]),
        "vrm_scene_set_completion_counter": (ci, [vp, vp]),
        "vrm_claim_next": (ci, [ci, vp, vp, vp]),
        "vrm_wait_flags_device": (ci, [ci, vp, vp, u32, u32, u32, u32, vp]),
        "vrm_render_views_sharded": (ci, [vp, u32, vp, u32, vp, u32, ci, u32, u32, vp, ci, vp, C.POINTER(f32)]),
        "vrm_scene_add_dense": (ci, [vp, vp, vp, vp, u32, C.POINTER(u64)]),
        "vrm_scene_add_dense_device": (ci, [vp, vp, vp, vp, u32, C.POINTER(u64)]),
        "vrm_scene_read_box": (ci, [vp, vp, vp, vp]),
        "vrm_scene_read_box_device": (ci, [vp, vp, vp, vp]),
        "vrm_scene_read_voxels": (ci, [vp, vp, vp, vp, vp, u64, C.POINTER(u64)]),
        "vrm_scene_read_voxels_device": (ci, [vp, vp, vp, vp, vp, u64, C.POINTER(u64)]),
        "vrm_hit_surface_views": (ci, [vp, vp, u32, vp, u32, u32, u32, vp, vp, vp]),
        "vrm_hit_surface_views_device": (ci, [vp, vp, u32, vp, u32, u32, u32, vp, vp, vp]),
        "vrm_hit_surface_rays": (ci, [vp, vp, u64, vp, u32, vp, vp, vp]),
        "vrm_hit_surface_rays_device": (ci, [vp, vp, u64, vp, u32, vp, vp, vp]),
        "vrm_cast_rays": (ci, [vp, vp, vp, u64, vp, u32, vp, vp, vp, vp]),
        "vrm_cast_rays_device": (ci, [vp, vp, vp, u64, vp, u32, vp, vp, vp, vp]),
        "vrm_cast_views": (ci, [vp, vp, u32, vp, u32, u32, u32, vp, vp, vp, vp]),
        "vrm_cast_views_device": (ci, [vp, vp, u32, vp, u32, u32, u32, vp, vp, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def device_available() -> bool:
    return bool(load_library().vrm_device_available())


def microbench_l2(device: int = 0, working_set_bytes: int = 32 << 20):
    """L2 roofs for an L2-resident working set: dict(gather8_loads_per_ns, gather8_gbs, stream_gbs).  Measurement only."""
    a, b, c = C.c_float(), C.c_float(), C.c_float()
    rc = load_library().vrm_microbench_l2(device, working_set_bytes, C.byref(a), C.byref(b), C.byref(c))
    if rc:
        raise VrmError(f"vrm_microbench_l2 failed: {rc}")
    return dict(working_set_bytes=working_set_bytes, gather8_loads_per_ns=a.value, gather8_gbs=b.value, stream_gbs=c.value)


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


def _f3(v):
    return np.ascontiguousarray(np.asarray(v, np.float32).reshape(3))


def _box(origin, dims):
    """(origin, dims) of a dense volume as the int32[3] / uint32[3] arrays of the C ABI."""
    o = np.ascontiguousarray(np.asarray(origin, np.int64).reshape(3))
    d = np.ascontiguousarray(np.asarray(dims, np.int64).reshape(3))
    if (d < 0).any() or (d >= 1 << 32).any() or (o < -(1 << 31)).any() or (o >= 1 << 31).any():
        raise ValueError(f"box out of range: origin {o.tolist()}, dims {d.tolist()}")
    return o.astype(np.int32), d.astype(np.uint32)


def make_unit_vector(v):
    out = np.zeros(3, np.float32)
    rc = load_library().vrm_make_unit_vector(_ptr(_f3(v)), _ptr(out))
    if rc:
        raise VrmError("vrm_make_unit_vector failed")
    return out


class Camera:
    """The reference's pinhole camera (Camera.cuh:11-23).  ``data`` is the 60-byte struct as 15 float32:
    origin, lowerLeftCorner, horizontalVector, verticalVector, forwardVector."""

    def __init__(self, origin, look_at, up=(0.0, 1.0, 0.0), field_of_view=60.0, aspect_ratio=1920.0 / 1080.0):
        self.data = np.zeros(15, np.float32)
        rc = load_library().vrm_camera_make(_ptr(_f3(origin)), _ptr(_f3(look_at)), _ptr(_f3(up)),
                                            C.c_float(np.float32(field_of_view)), C.c_float(np.float32(aspect_ratio)), _ptr(self.data))
        if rc:
            raise VrmError("vrm_camera_make failed")

    @staticmethod
    def reference_default(width=1920, height=1080):
        """main/Main.cu:195-199."""
        return Camera((6.0, 2.0, 6.0), (0.0, 0.0, -1.0), (0.0, 1.0, 0.0), 60.0, np.float32(width) / np.float32(height))


class VoxelScene:
    """One scene on one GPU (one handle = one device + one stream)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        self.h = C.c_void_p()
        rc = self.lib.vrm_scene_create(device, C.byref(self.h))
        if rc:
            self.h = C.c_void_p()
            raise VrmError(f"vrm_scene_create(device={device}) failed: {self.lib.vrm_error_string(rc).decode()} "
                           "(a CUDA device is required; there is no CPU fallback)")
        self.device = device
        self.storage = None
        self.build_ms = None

    # -- plumbing ------------------------------------------------------------------------------------------------
    def _check(self, rc, what):
        if rc:
            raise VrmError(f"{what}: {self.lib.vrm_error_string(rc).decode()}: {self.lib.vrm_last_error(self.h).decode()}")

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.lib.vrm_scene_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_ptr: int):
        """Run on the caller's cudaStream_t (0 = the legacy default stream)."""
        self._check(self.lib.vrm_scene_set_stream(self.h, C.c_void_p(cuda_stream_ptr)), "vrm_scene_set_stream")

    def reset_stream(self):
        self._check(self.lib.vrm_scene_reset_stream(self.h), "vrm_scene_reset_stream")

    def synchronize(self):
        self._check(self.lib.vrm_scene_synchronize(self.h), "vrm_scene_synchronize")

    # -- scene construction --------------------------------------------------------------------------------------
    def insert_voxel(self, x: int, y: int, z: int, color: int):
        """``VoxelSceneCPU::insertVoxel``: one voxel per call (collected on the host by the library, no device work per call)."""
        rc = self.lib.vrm_scene_insert_voxel(self.h, x, y, z, color)
        if rc:
            self._check(rc, "vrm_scene_insert_voxel")

    def add_voxels(self, xyz, rgb):
        xyz = np.ascontiguousarray(xyz, np.int32).reshape(-1, 3)
        rgb = np.ascontiguousarray(rgb, np.uint32).reshape(-1)
        if xyz.shape[0] != rgb.shape[0]:
            raise ValueError("xyz and rgb disagree on the voxel count")
        self._check(self.lib.vrm_scene_add_voxels(self.h, _ptr(xyz), _ptr(rgb), xyz.shape[0]), "vrm_scene_add_voxels")

    def add_voxels_device(self, d_xyz_ptr: int, d_rgb_ptr: int, n: int):
        self._check(self.lib.vrm_scene_add_voxels_device(self.h, C.c_void_p(d_xyz_ptr), C.c_void_p(d_rgb_ptr), n), "vrm_scene_add_voxels_device")

    def add_dense(self, volume, origin=(0, 0, 0), empty_value: int = EMPTY) -> int:
        """Append every cell of ``volume`` (uint32, shape (nx, ny, nz), indexed [x][y][z]: cell [i, j, k] is the voxel at
        origin + (i, j, k)) whose value is not ``empty_value``, in C order, the value as its colour -- the same list
        ``add_voxels`` of those voxels in that order would append.  Returns the number of voxels added."""
        vol = np.asarray(volume)
        if vol.dtype != np.uint32 or vol.ndim != 3:
            raise ValueError("add_dense takes a 3-D uint32 volume")
        vol = np.ascontiguousarray(vol)
        o, d = _box(origin, vol.shape)
        n = C.c_uint64()
        self._check(self.lib.vrm_scene_add_dense(self.h, _ptr(vol), _ptr(d), _ptr(o), int(empty_value), C.byref(n)), "vrm_scene_add_dense")
        return int(n.value)

    def add_dense_device(self, d_ptr: int, dims, origin=(0, 0, 0), empty_value: int = EMPTY) -> int:
        """``add_dense`` of a C-contiguous uint32 volume in device memory (4-byte aligned), e.g. ``tensor.data_ptr()``.  Enqueued
        on the scene's stream after one synchronisation to learn the count; the volume must stay valid until that work has run."""
        o, d = _box(origin, dims)
        n = C.c_uint64()
        self._check(self.lib.vrm_scene_add_dense_device(self.h, C.c_void_p(d_ptr), _ptr(d), _ptr(o), int(empty_value), C.byref(n)),
                    "vrm_scene_add_dense_device")
        return int(n.value)

    def read_box(self, origin, dims):
        """The box ``[origin, origin + dims)`` of the built scene as a uint32 volume of shape ``dims`` (indexed [x][y][z]): the
        colour of every cell, or ``EMPTY`` -- what ``lookup`` returns for the cell's coordinate."""
        o, d = _box(origin, dims)
        out = np.empty(tuple(int(v) for v in d), np.uint32)
        self._check(self.lib.vrm_scene_read_box(self.h, _ptr(o), _ptr(d), _ptr(out)), "vrm_scene_read_box")
        return out

    def read_box_device(self, origin, dims, d_out_ptr: int):
        """``read_box`` into a device buffer of prod(dims) uint32 (4-byte aligned); asynchronous on the scene's stream."""
        o, d = _box(origin, dims)
        self._check(self.lib.vrm_scene_read_box_device(self.h, _ptr(o), _ptr(d), C.c_void_p(d_out_ptr)), "vrm_scene_read_box_device")

    def _voxel_box(self, origin, dims):
        if origin is None and dims is None:
            origin, dims = self.scene_box()
        elif origin is None or dims is None:
            raise ValueError("give both origin and dims, or neither (the whole scene_box())")
        return _box(origin, dims)

    def count_voxels(self, origin=None, dims=None) -> int:
        """Number of stored voxels in the box ``[origin, origin + dims)`` (default: ``scene_box()``, whose count is ``unique_voxels``)."""
        o, d = self._voxel_box(origin, dims)
        n = C.c_uint64()
        self._check(self.lib.vrm_scene_read_voxels(self.h, _ptr(o), _ptr(d), None, None, 0, C.byref(n)), "vrm_scene_read_voxels")
        return int(n.value)

    def read_voxels(self, origin=None, dims=None):
        """The stored voxels of the box ``[origin, origin + dims)`` (default: ``scene_box()``) as ``(xyz int32 (n, 3), rgb uint32 (n,))``
        sorted by (x, y, z), z fastest: the non-``EMPTY`` cells of ``read_box`` in C order, plus any voxel stored with the colour ``EMPTY``.
        The same arrays ``add_voxels`` takes, so ``other.add_voxels(*scene.read_voxels())`` rebuilds the scene."""
        o, d = self._voxel_box(origin, dims)
        n = self.count_voxels(o, d)
        xyz = np.empty((n, 3), np.int32)
        rgb = np.empty(n, np.uint32)
        got = C.c_uint64()
        if n:
            self._check(self.lib.vrm_scene_read_voxels(self.h, _ptr(o), _ptr(d), _ptr(xyz), _ptr(rgb), n, C.byref(got)), "vrm_scene_read_voxels")
            assert got.value == n
        return xyz, rgb

    def read_voxels_device(self, origin, dims, d_xyz_ptr: int, d_rgb_ptr: int, capacity: int) -> int:
        """``read_voxels`` into device buffers of ``capacity`` voxels (n x 3 int32 and n uint32, 4-byte aligned), e.g. torch tensors.
        Returns the count after one synchronisation; the voxels are written in stream order on the scene's stream.  A capacity below the
        count raises and writes nothing; ``count_voxels`` sizes the buffers."""
        o, d = _box(origin, dims)
        n = C.c_uint64()
        self._check(self.lib.vrm_scene_read_voxels_device(self.h, _ptr(o), _ptr(d), C.c_void_p(d_xyz_ptr), C.c_void_p(d_rgb_ptr), int(capacity),
                                                          C.byref(n)), "vrm_scene_read_voxels_device")
        return int(n.value)

    def scene_box(self):
        """(origin, dims) of the box the built scene's region table covers: every stored voxel lies inside it."""
        info = self.info()
        return (64 * info["min_coord"],) * 3, (64 * info["diameter"],) * 3

    def generate_terrain(self, size: int = 512, seed: int = 1234, max_height: int = 0) -> int:
        """``scenes.terrain(size, seed, max_height)`` generated on the GPU straight into the staging list; returns the voxel count."""
        n = C.c_uint64()
        self._check(self.lib.vrm_scene_generate_terrain(self.h, size, seed, max_height, C.byref(n)), "vrm_scene_generate_terrain")
        return int(n.value)

    def generate_sparse_shells(self, size: int = 1024, cell: int = 64, seed: int = 7, fill_pct: int = 35) -> int:
        """``scenes.sparse_shells(size, cell, seed, fill_pct)`` generated on the GPU straight into the staging list."""
        n = C.c_uint64()
        self._check(self.lib.vrm_scene_generate_sparse_shells(self.h, size, cell, seed, fill_pct, C.byref(n)), "vrm_scene_generate_sparse_shells")
        return int(n.value)

    def generate_cube(self, x: int, y: int, z: int, half_width: int) -> int:
        """``VoxelCube::generateVoxelCube`` (= ``scenes.hollow_cube``) on the GPU, in the reference's insertion order."""
        n = C.c_uint64()
        self._check(self.lib.vrm_scene_generate_cube(self.h, x, y, z, half_width, C.byref(n)), "vrm_scene_generate_cube")
        return int(n.value)

    def generate_sphere(self, x: int, y: int, z: int, radius: int, checkered: bool = False) -> int:
        """``VoxelSphere::generate[Checkered]VoxelSphere`` (= ``scenes.sphere_shell``) on the GPU, in the reference's insertion order."""
        n = C.c_uint64()
        self._check(self.lib.vrm_scene_generate_sphere(self.h, x, y, z, radius, int(checkered), C.byref(n)), "vrm_scene_generate_sphere")
        return int(n.value)

    def generate_voxel_scene(self, storage_type):
        st = STORAGE[storage_type] if isinstance(storage_type, str) else int(storage_type)
        ms = C.c_float()
        self._check(self.lib.vrm_scene_build(self.h, st, C.byref(ms)), "vrm_scene_build")
        self.storage = st
        self.build_ms = ms.value
        return ms.value

    def info(self):
        d, m, f, u, b = C.c_uint32(), C.c_int32(), C.c_uint32(), C.c_uint64(), C.c_uint64()
        self._check(self.lib.vrm_scene_info(self.h, C.byref(d), C.byref(m), C.byref(f), C.byref(u), C.byref(b)), "vrm_scene_info")
        return dict(diameter=d.value, min_coord=m.value, filled=f.value, unique_voxels=u.value, bytes=b.value)

    def get_array_diameter(self):
        return self.info()["diameter"]

    def get_array_size(self):
        return self.info()["diameter"] ** 3

    def get_min_coord(self):
        return self.info()["min_coord"]

    # -- lighting ------------------------------------------------------------------------------------------------
    def setup_constant_values(self, light_direction=None, light_color=(1.0, 1.0, 1.0), light_position=(10.0, 10.0, -10.0),
                              use_point_light=False, use_shadows=True):
        if light_direction is None:
            light_direction = make_unit_vector((1.0, 1.0, 1.0))
        self._check(self.lib.vrm_set_lighting(self.h, _ptr(_f3(light_direction)), _ptr(_f3(light_color)), _ptr(_f3(light_position)),
                                              int(use_point_light), int(use_shadows)), "vrm_set_lighting")

    # -- rendering -----------------------------------------------------------------------------------------------
    @staticmethod
    def _algo(algorithm):
        return ALGORITHM[algorithm] if isinstance(algorithm, str) else int(algorithm)

    @staticmethod
    def _cam(camera):
        return np.ascontiguousarray(camera.data if isinstance(camera, Camera) else camera, np.float32)

    def run_raymarching_kernel(self, width, height, algorithm, camera, scale=1, translation=(0.0, 0.0, 0.0), want_hits=False,
                               rgb_out=None, want_surface=False):
        """Render one frame into host memory.  Returns dict(rgb[H,W,3] uint8, hits[H,W,4] int32 | None, kernel_ms); with
        ``want_surface`` also depth[H,W] float32 and face[H,W] uint8 of ``hit_surface_views`` (the hit map is then rendered internally)."""
        rgb = rgb_out if rgb_out is not None else np.zeros((height, width, 3), np.uint8)
        hits = np.zeros((height, width, 4), np.int32) if want_hits or want_surface else None
        ms = C.c_float()
        cam = self._cam(camera)
        self._check(self.lib.vrm_render(self.h, _ptr(cam), _ptr(_f3(translation)), scale, self._algo(algorithm), width, height,
                                        _ptr(rgb), _ptr(hits), C.byref(ms)), "vrm_render")
        out = dict(rgb=rgb, hits=hits if want_hits else None, kernel_ms=ms.value)
        if want_surface:
            depth, face = self.hit_surface_views(hits, [cam], width, height, scale, translation)
            out.update(depth=depth[0], face=face[0])
        return out

    render = run_raymarching_kernel

    def render_device(self, width, height, algorithm, camera, d_rgb_ptr: int, d_hits_ptr: int | None = None, scale=1,
                      translation=(0.0, 0.0, 0.0)):
        cam = self._cam(camera)
        self._check(self.lib.vrm_render_device(self.h, _ptr(cam), _ptr(_f3(translation)), scale, self._algo(algorithm), width, height,
                                               C.c_void_p(d_rgb_ptr), C.c_void_p(d_hits_ptr or 0)), "vrm_render_device")

    def render_views_device(self, width, height, algorithm, cameras, d_rgb_ptr: int, d_hits_ptr: int | None = None, scale=1,
                            translation=(0.0, 0.0, 0.0), view_stride: int = 1):
        """All ``cameras`` in one launch; view ``v`` goes to frame slot ``v * view_stride`` of the outputs."""
        cams = np.ascontiguousarray(np.stack([self._cam(c) for c in cameras]), np.float32)
        self._check(self.lib.vrm_render_views_device_strided(self.h, _ptr(cams), cams.shape[0], _ptr(_f3(translation)), scale, self._algo(algorithm),
                                                             width, height, C.c_void_p(d_rgb_ptr), C.c_void_p(d_hits_ptr or 0), int(view_stride)),
                    "vrm_render_views_device_strided")

    def render_views(self, width, height, algorithm, cameras, scale=1, translation=(0.0, 0.0, 0.0), rgb_out=None):
        """A batch of views (camera orbit) into host frames ``[n, H, W, 3]``; ``rgb_out`` may be a pinned buffer (written directly
        by the kernel) or pageable memory (double-buffered device batches, copies overlapped with rendering)."""
        cams = np.ascontiguousarray(np.stack([self._cam(c) for c in cameras]).astype(np.float32))
        n = cams.shape[0]
        if rgb_out is None:
            rgb_out = np.zeros((n, height, width, 3), np.uint8)
        assert rgb_out.dtype == np.uint8 and rgb_out.size == n * height * width * 3 and rgb_out.flags["C_CONTIGUOUS"]
        ms = C.c_float()
        self._check(self.lib.vrm_render_views(self.h, _ptr(cams), n, _ptr(_f3(translation)), int(scale), self._algo(algorithm), width, height,
                                              _ptr(rgb_out), C.byref(ms)), "vrm_render_views")
        return {"rgb": rgb_out.reshape(n, height, width, 3), "total_ms": ms.value}

    def trace_rays(self, rays, algorithm, scale=1, translation=(0.0, 0.0, 0.0), want_hits=False, want_surface=False):
        """Trace world rays (n, 6).  Returns dict(colour (n,) uint32, hits (n, 4) int32 | None, kernel_ms); with ``want_surface`` also
        depth (n,) float32 and face (n,) uint8 of ``hit_surface_rays`` (the hit records are then traced internally)."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 6)
        n = rays.shape[0]
        colour = np.zeros(n, np.uint32)
        hits = np.zeros((n, 4), np.int32) if want_hits or want_surface else None
        ms = C.c_float()
        self._check(self.lib.vrm_trace_rays(self.h, _ptr(rays), n, _ptr(_f3(translation)), scale, self._algo(algorithm), _ptr(colour),
                                            _ptr(hits), C.byref(ms)), "vrm_trace_rays")
        out = dict(colour=colour, hits=hits if want_hits else None, kernel_ms=ms.value)
        if want_surface:
            out["depth"], out["face"] = self.hit_surface_rays(hits, rays, scale, translation)
        return out

    def trace_rays_device(self, d_rays_ptr: int, n: int, algorithm, d_colour_ptr: int, d_hits_ptr: int | None = None, scale=1,
                          translation=(0.0, 0.0, 0.0)):
        self._check(self.lib.vrm_trace_rays_device(self.h, C.c_void_p(d_rays_ptr), n, _ptr(_f3(translation)), scale, self._algo(algorithm),
                                                   C.c_void_p(d_colour_ptr), C.c_void_p(d_hits_ptr or 0)), "vrm_trace_rays_device")

    # -- hit surfaces (include/vrm_b200.h "hit surfaces": depth and entered face from a hit map and the exact ray) -----------------
    def hit_surface_views(self, hits, cameras, width, height, scale=1, translation=(0.0, 0.0, 0.0)):
        """Depth and face of a view-major hit map ``hits`` (n, H, W, 4) int32 as ``render`` / ``render_views_device`` write it, for the
        n ``cameras`` it was rendered with.  Returns (depth (n, H, W) float32, face (n, H, W) uint8): depth = world distance from the
        camera origin along the pixel's ray (+inf for a miss), face = 1..6 for -x, +x, -y, +y, -z, +z (``FACE_NORMALS``), 0 for a miss."""
        cams = np.ascontiguousarray(np.stack([self._cam(c) for c in cameras]), np.float32)
        n = cams.shape[0]
        hits = np.ascontiguousarray(hits, np.int32)
        if hits.size != n * height * width * 4:
            raise ValueError(f"hits holds {hits.size // 4} records, {n} views of {width}x{height} need {n * height * width}")
        depth = np.empty((n, height, width), np.float32)
        face = np.empty((n, height, width), np.uint8)
        self._check(self.lib.vrm_hit_surface_views(self.h, _ptr(cams), n, _ptr(_f3(translation)), int(scale), width, height, _ptr(hits),
                                                   _ptr(depth), _ptr(face)), "vrm_hit_surface_views")
        return depth, face

    def hit_surface_views_device(self, d_hits_ptr: int, cameras, width, height, d_depth_ptr: int | None, d_face_ptr: int | None, scale=1,
                                 translation=(0.0, 0.0, 0.0)):
        """``hit_surface_views`` on device buffers (e.g. ``tensor.data_ptr()``; hits 16-byte aligned, depth 4-byte aligned; either output
        may be None); asynchronous on the scene's stream."""
        cams = np.ascontiguousarray(np.stack([self._cam(c) for c in cameras]), np.float32)
        self._check(self.lib.vrm_hit_surface_views_device(self.h, _ptr(cams), cams.shape[0], _ptr(_f3(translation)), int(scale), width, height,
                                                          C.c_void_p(d_hits_ptr), C.c_void_p(d_depth_ptr or 0), C.c_void_p(d_face_ptr or 0)),
                    "vrm_hit_surface_views_device")

    def hit_surface_rays(self, hits, rays, scale=1, translation=(0.0, 0.0, 0.0)):
        """Depth and face of traced rays (n, 6) and their hit records (n, 4) from ``trace_rays``.  Returns (depth (n,) float32, face (n,)
        uint8): depth = world ray parameter of the entry point (origin + depth * direction), +inf for a miss."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 6)
        n = rays.shape[0]
        hits = np.ascontiguousarray(hits, np.int32)
        if hits.size != n * 4:
            raise ValueError(f"hits holds {hits.size // 4} records for {n} rays")
        depth = np.empty(n, np.float32)
        face = np.empty(n, np.uint8)
        self._check(self.lib.vrm_hit_surface_rays(self.h, _ptr(rays), n, _ptr(_f3(translation)), int(scale), _ptr(hits), _ptr(depth), _ptr(face)),
                    "vrm_hit_surface_rays")
        return depth, face

    def hit_surface_rays_device(self, d_hits_ptr: int, d_rays_ptr: int, n: int, d_depth_ptr: int | None, d_face_ptr: int | None, scale=1,
                                translation=(0.0, 0.0, 0.0)):
        """``hit_surface_rays`` on device buffers (hits 16-byte aligned, rays and depth 4-byte aligned); asynchronous on the scene's stream."""
        self._check(self.lib.vrm_hit_surface_rays_device(self.h, C.c_void_p(d_rays_ptr), int(n), _ptr(_f3(translation)), int(scale),
                                                         C.c_void_p(d_hits_ptr), C.c_void_p(d_depth_ptr or 0), C.c_void_p(d_face_ptr or 0)),
                    "vrm_hit_surface_rays_device")

    # -- exact ray casts (include/vrm_b200.h "exact ray casts": first stored voxel along the exact ray within an interval) -----------
    def cast_rays(self, rays, ranges=None, scale=1, translation=(0.0, 0.0, 0.0)):
        """The first stored voxel along each exact world ray (n, 6) within its interval ``ranges`` (n, 2) {t_near, t_far} (None: [0, +inf)).
        Returns dict(hits (n, 4) int32 {x, y, z, 1 | 0}, depth (n,) float32 world ray parameter of the entry (t_near for a hit in the start
        cell, +inf for a miss), face (n,) uint8 1..6 of the entered face (``FACE_NORMALS``; 0 in the start cell or for a miss),
        colour (n,) uint32 the stored colour (``EMPTY`` for a miss))."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 6)
        n = rays.shape[0]
        rg = None
        if ranges is not None:
            rg = np.ascontiguousarray(ranges, np.float32).reshape(-1, 2)
            if rg.shape[0] != n:
                raise ValueError(f"ranges holds {rg.shape[0]} intervals for {n} rays")
        out = dict(hits=np.empty((n, 4), np.int32), depth=np.empty(n, np.float32), face=np.empty(n, np.uint8), colour=np.empty(n, np.uint32))
        self._check(self.lib.vrm_cast_rays(self.h, _ptr(rays), _ptr(rg), n, _ptr(_f3(translation)), int(scale), _ptr(out["hits"]),
                                           _ptr(out["depth"]), _ptr(out["face"]), _ptr(out["colour"])), "vrm_cast_rays")
        return out

    def cast_rays_device(self, d_rays_ptr: int, n: int, d_ranges_ptr: int | None = None, d_hits_ptr: int | None = None, d_depth_ptr: int | None = None,
                         d_face_ptr: int | None = None, d_colour_ptr: int | None = None, scale=1, translation=(0.0, 0.0, 0.0)):
        """``cast_rays`` on device buffers (rays, ranges, depth, colour 4-byte aligned, hits 16-byte aligned; each output optional, not all);
        asynchronous on the scene's stream."""
        self._check(self.lib.vrm_cast_rays_device(self.h, C.c_void_p(d_rays_ptr), C.c_void_p(d_ranges_ptr or 0), int(n), _ptr(_f3(translation)),
                                                  int(scale), C.c_void_p(d_hits_ptr or 0), C.c_void_p(d_depth_ptr or 0), C.c_void_p(d_face_ptr or 0),
                                                  C.c_void_p(d_colour_ptr or 0)), "vrm_cast_rays_device")

    def cast_views(self, cameras, width, height, scale=1, translation=(0.0, 0.0, 0.0)):
        """``cast_rays`` for the pixel rays of each camera's frame (the render's rays, over [0, +inf)), view-major: hits (n, H, W, 4),
        depth (n, H, W) = world distance from the camera origin along the pixel's ray, face and colour (n, H, W)."""
        cams = np.ascontiguousarray(np.stack([self._cam(c) for c in cameras]), np.float32)
        v = cams.shape[0]
        out = dict(hits=np.empty((v, height, width, 4), np.int32), depth=np.empty((v, height, width), np.float32),
                   face=np.empty((v, height, width), np.uint8), colour=np.empty((v, height, width), np.uint32))
        self._check(self.lib.vrm_cast_views(self.h, _ptr(cams), v, _ptr(_f3(translation)), int(scale), width, height, _ptr(out["hits"]),
                                            _ptr(out["depth"]), _ptr(out["face"]), _ptr(out["colour"])), "vrm_cast_views")
        return out

    def cast_views_device(self, cameras, width, height, d_hits_ptr: int | None = None, d_depth_ptr: int | None = None, d_face_ptr: int | None = None,
                          d_colour_ptr: int | None = None, scale=1, translation=(0.0, 0.0, 0.0)):
        """``cast_views`` into device buffers (alignment as ``cast_rays_device``); asynchronous on the scene's stream."""
        cams = np.ascontiguousarray(np.stack([self._cam(c) for c in cameras]), np.float32)
        self._check(self.lib.vrm_cast_views_device(self.h, _ptr(cams), cams.shape[0], _ptr(_f3(translation)), int(scale), width, height,
                                                   C.c_void_p(d_hits_ptr or 0), C.c_void_p(d_depth_ptr or 0), C.c_void_p(d_face_ptr or 0),
                                                   C.c_void_p(d_colour_ptr or 0)), "vrm_cast_views_device")

    def lookup(self, xyz):
        xyz = np.ascontiguousarray(xyz, np.int32).reshape(-1, 3)
        n = xyz.shape[0]
        out = np.zeros(n, np.uint32)
        exists = np.zeros(n, np.uint8)
        self._check(self.lib.vrm_lookup(self.h, _ptr(xyz), n, _ptr(out), _ptr(exists)), "vrm_lookup")
        return out, exists

    def set_completion_flag(self, d_flag_ptr: int | None, first_value: int = 1):
        """Every later render launch of this scene stores first_value, first_value + 1, ... into the word at ``d_flag_ptr`` (device or
        peer memory) behind its frame (``multigpu.PeerFrameBuffer.flag_ptr``); ``None`` switches the signal off."""
        self._check(self.lib.vrm_scene_set_completion_flag(self.h, C.c_void_p(d_flag_ptr or 0), first_value), "vrm_scene_set_completion_flag")

    def set_completion_counter(self, d_counter_ptr: int | None):
        """Counting form of the completion signal: every render launch adds its number of views to the word at ``d_counter_ptr``."""
        self._check(self.lib.vrm_scene_set_completion_counter(self.h, C.c_void_p(d_counter_ptr or 0)), "vrm_scene_set_completion_counter")

    # -- statistics ----------------------------------------------------------------------------------------------
    def set_l2_persistence(self, enabled: bool):
        self._check(self.lib.vrm_set_l2_persistence(self.h, int(enabled)), "vrm_set_l2_persistence")

    def set_statistics(self, enabled: bool, as_executed: bool = False):
        """Event counters for the next render / trace calls.  Default: comparable with the reference's (every shadow ray is traced, as
        the reference does).  ``as_executed``: the counters of the work the production kernels do -- a shadow ray whose pixel is already
        black (normal facing away from the light: colour * !shadow = 0 either way) is not traced."""
        self._check(self.lib.vrm_set_statistics(self.h, (2 if as_executed else 1) if enabled else 0), "vrm_set_statistics")

    def get_statistics(self):
        out = np.zeros(8, np.uint64)
        self._check(self.lib.vrm_get_statistics(self.h, _ptr(out)), "vrm_get_statistics")
        keys = ["exist_checks", "exist_false", "lookups", "lookup_hits", "table2_probes", "region_reads", "rays", "crawl_skipped"]
        return {k: int(v) for k, v in zip(keys, out)}


def render_views_sharded(scene_list, width, height, algorithm, cameras, scale=1, translation=(0.0, 0.0, 0.0), rgb_out=None, d_rgb_ptr: int | None = None):
    """``vrm_render_views_sharded``: ONE process, one built ``VoxelScene`` per device (same voxels); the views are claimed dynamically
    and gathered on the first scene's device.  Returns dict(rgb[n,H,W,3] | None, views_per_scene, total_ms); with ``d_rgb_ptr`` the
    frames stay in that device buffer (on the first scene's device)."""
    lib = load_library()
    cams = np.ascontiguousarray(np.stack([VoxelScene._cam(c) for c in cameras]).astype(np.float32))
    n = cams.shape[0]
    handles = (C.c_void_p * len(scene_list))(*[s.h for s in scene_list])
    counts = np.zeros(len(scene_list), np.uint32)
    ms = C.c_float()
    on_device = d_rgb_ptr is not None
    if not on_device:
        if rgb_out is None:
            rgb_out = np.zeros((n, height, width, 3), np.uint8)
        assert rgb_out.dtype == np.uint8 and rgb_out.size == n * height * width * 3 and rgb_out.flags["C_CONTIGUOUS"]
    out = C.c_void_p(d_rgb_ptr) if on_device else _ptr(rgb_out)
    rc = lib.vrm_render_views_sharded(C.cast(handles, C.c_void_p), len(scene_list), _ptr(cams), n, _ptr(_f3(translation)), int(scale),
                                      VoxelScene._algo(algorithm), width, height, out, int(on_device), _ptr(counts), C.byref(ms))
    if rc:
        raise VrmError(f"vrm_render_views_sharded: {lib.vrm_error_string(rc).decode()}: {lib.vrm_last_error(scene_list[0].h).decode()}")
    return dict(rgb=None if on_device else rgb_out.reshape(n, height, width, 3), views_per_scene=counts.tolist(), total_ms=ms.value)
