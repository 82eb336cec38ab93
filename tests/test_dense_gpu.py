"""GPU tier: dense uint32 volumes in and out of a scene (vrm_scene_add_dense[_device], vrm_scene_read_box[_device]).

A dense volume of dims (nx, ny, nz) at origin o is indexed [x][y][z]: cell [i, j, k] is the voxel at o + (i, j, k).  add_dense must
append exactly the list add_voxels of the non-empty cells in C order appends (last insert wins across call kinds), and read_box must
return, cell for cell, what vrm_lookup returns.  Both are checked bit for bit against the oracle and against the list path, for
both storage types."""
import ctypes as C

import numpy as np
import pytest

from tests.common import COMBOS, build_oracle, lookup_queries, oracle_kind, po, scenes
from voxelraymarcher_b200 import api

pytestmark = pytest.mark.gpu

STORAGES = ["hashtable", "vcs"]
VOL_SHAPE, VOL_ORIGIN = (150, 97, 130), (-70, -5, 33)   # negative, several regions, not cluster-aligned
MARGIN = 80                                             # the read box crosses region-table edges (x at -128, z at 192)


def random_volume(shape, seed, occupancy=0.1, empty=api.EMPTY):
    rng = np.random.default_rng(seed)
    vol = np.full(shape, empty, np.uint32)
    mask = rng.random(shape) < occupancy
    vol[mask] = rng.integers(1, 1 << 24, int(mask.sum()), dtype=np.uint32)
    return vol


def voxels_of(vol, origin, empty=api.EMPTY):
    """The non-empty cells of a volume as a voxel list, in C order."""
    mask = vol != empty
    return (np.argwhere(mask) + np.asarray(origin)).astype(np.int32), vol[mask].astype(np.uint32)


def box_cells(origin, dims):
    """Every coordinate of a box in C order (x slowest, z fastest)."""
    g = np.meshgrid(*[np.arange(o, o + d, dtype=np.int32) for o, d in zip(origin, dims)], indexing="ij")
    return np.ascontiguousarray(np.stack([a.ravel() for a in g], 1))


def to_device(vol):
    import torch
    return torch.from_numpy(np.ascontiguousarray(vol).view(np.int32)).cuda()


def read_box_device(s, origin, dims):
    import torch
    out = torch.empty(tuple(dims), dtype=torch.int32, device="cuda")
    s.read_box_device(origin, dims, out.data_ptr())
    s.synchronize()
    return out.cpu().numpy().view(np.uint32)


def grown(vol, margin, fill=api.EMPTY):
    big = np.full(tuple(d + 2 * margin for d in vol.shape), fill, np.uint32)
    big[margin:margin + vol.shape[0], margin:margin + vol.shape[1], margin:margin + vol.shape[2]] = vol
    return big


@pytest.fixture(scope="module")
def volume():
    return random_volume(VOL_SHAPE, seed=2024)


@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("variant", ["host", "device"])
@pytest.mark.parametrize("empty", ["default", "zero"])
def test_round_trip(volume, storage, variant, empty):
    vol = volume if empty == "default" else np.where(volume == api.EMPTY, 0, volume).astype(np.uint32)
    ev = api.EMPTY if empty == "default" else 0
    n_expected = int((volume != api.EMPTY).sum())
    s = api.VoxelScene(0)
    if variant == "host":
        n = s.add_dense(vol, VOL_ORIGIN, empty_value=ev)
    else:
        d_vol = to_device(vol)
        n = s.add_dense_device(d_vol.data_ptr(), vol.shape, VOL_ORIGIN, empty_value=ev)
    assert n == n_expected
    s.generate_voxel_scene(storage)
    assert s.info()["unique_voxels"] == n_expected
    origin = tuple(o - MARGIN for o in VOL_ORIGIN)
    dims = tuple(d + 2 * MARGIN for d in VOL_SHAPE)
    got = s.read_box(origin, dims) if variant == "host" else read_box_device(s, origin, dims)
    assert got.shape == dims and got.dtype == np.uint32
    assert np.array_equal(got, grown(volume, MARGIN))
    # 1x1x1 boxes: stored voxels, empty cells, cells outside the table
    xyz, rgb = voxels_of(volume, VOL_ORIGIN)
    picks = np.concatenate([xyz[:: max(1, len(xyz) // 40)], np.array([[-70, -5, 32], [200, 0, 0], [-129, 0, 100], [0, 0, 0]], np.int32)])
    want = s.lookup(picks)[0]
    for p, w in zip(picks, want):
        one = s.read_box(p, (1, 1, 1)) if variant == "host" else read_box_device(s, p, (1, 1, 1))
        assert one.shape == (1, 1, 1) and int(one[0, 0, 0]) == int(w), (p, one, w)
    # a box entirely outside the region table, and one near the end of the int32 range
    assert (s.read_box((1000, -2000, 300), (7, 5, 33)) == api.EMPTY).all()
    assert (s.read_box((2**31 - 9, 0, -(2**31)), (8, 3, 40)) == api.EMPTY).all()


@pytest.mark.parametrize("storage,algo", COMBOS)
def test_same_scene_as_the_list_path(volume, storage, algo):
    xyz, rgb = voxels_of(volume, VOL_ORIGIN)
    kind = oracle_kind()
    po.set_lighting(kind)
    ref = build_oracle(kind, xyz, rgb, storage)
    dense = api.VoxelScene(0)
    dense.add_dense(volume, VOL_ORIGIN)
    dense.generate_voxel_scene(storage)
    listed = api.VoxelScene(0)
    listed.add_voxels(xyz, rgb)
    listed.generate_voxel_scene(storage)
    perm = np.random.default_rng(3).permutation(len(xyz))
    shuffled = api.VoxelScene(0)
    shuffled.add_voxels(xyz[perm], rgb[perm])
    shuffled.generate_voxel_scene(storage)
    info = dense.info()
    assert info == listed.info() == shuffled.info()
    assert dict(diameter=info["diameter"], min_coord=info["min_coord"], filled=info["filled"]) == ref.info()
    q = lookup_queries(xyz, 50000, seed=17)
    val, ex = dense.lookup(q)
    rval, rex = ref.lookup(q)
    assert np.array_equal(val, rval) and np.array_equal(ex, rex)
    assert np.array_equal(val, listed.lookup(q)[0]) and np.array_equal(val, shuffled.lookup(q)[0])
    centre = tuple(o + d / 2 for o, d in zip(VOL_ORIGIN, VOL_SHAPE))
    views = [((230.0, 160.0, 320.0), centre, 60.0), ((-260.0, 90.0, -140.0), centre, 50.0), ((5.0, 43.0, 98.0), (90.0, 10.0, 200.0), 70.0),
             ((40.0, 400.0, -30.0), centre, 35.0)]
    w, h = 320, 180
    for o, look, fov in views:
        cam = api.Camera(o, look, (0.0, 1.0, 0.0), fov, np.float32(w) / np.float32(h))
        got = dense.render(w, h, algo, cam, want_hits=True)
        want = ref.render(cam.data, w, h, algo)
        assert np.array_equal(got["hits"], want["hits"]), (storage, algo, o, int((got["hits"] != want["hits"]).any(-1).sum()))
        assert np.array_equal(got["rgb"], want["rgb"]), (storage, algo, o)
        assert want["hits"][..., 3].any()


@pytest.mark.parametrize("storage", STORAGES)
def test_insertion_order_across_call_kinds(storage):
    """add_voxels, then an overlapping add_dense, then an overlapping add_voxels: the last insert wins, whatever the call."""
    rng = np.random.default_rng(9)
    a_xyz = rng.integers(-20, 40, (30000, 3)).astype(np.int32)
    a_rgb = rng.integers(1, 1 << 24, 30000, dtype=np.uint32)
    vol = random_volume((40, 30, 50), seed=10, occupancy=0.3)
    v_origin = (-10, -3, 20)
    c_xyz = rng.integers(-20, 40, (20000, 3)).astype(np.int32)
    c_rgb = rng.integers(1, 1 << 24, 20000, dtype=np.uint32)
    s = api.VoxelScene(0)
    s.add_voxels(a_xyz, a_rgb)
    s.add_dense(vol, v_origin)
    s.add_voxels(c_xyz, c_rgb)
    s.generate_voxel_scene(storage)
    b_xyz, b_rgb = voxels_of(vol, v_origin)
    ref = build_oracle(oracle_kind(), np.concatenate([a_xyz, b_xyz, c_xyz]), np.concatenate([a_rgb, b_rgb, c_rgb]), storage)
    origin, dims = s.scene_box()
    got = s.read_box(origin, dims)
    want = ref.lookup(box_cells(origin, dims))[0].reshape(dims)
    assert np.array_equal(got, want)
    # the overlap really decides: some cells of the volume were overwritten by the later list, some overwrote the earlier one
    vx = got[b_xyz[:, 0] - origin[0], b_xyz[:, 1] - origin[1], b_xyz[:, 2] - origin[2]]
    assert (vx != b_rgb).any() and (vx == b_rgb).any()


@pytest.mark.parametrize("name", ["probe", "mini"])
def test_read_box_equals_lookup(name):
    xyz, rgb = scenes.probe_scene() if name == "probe" else scenes.mini_scene()
    boxes = {}
    for storage in STORAGES:
        s = api.VoxelScene(0)
        s.add_voxels(xyz, rgb)
        s.generate_voxel_scene(storage)
        origin, dims = s.scene_box()
        got = s.read_box(origin, dims)
        assert np.array_equal(got, s.lookup(box_cells(origin, dims))[0].reshape(dims)), storage
        assert np.array_equal(read_box_device(s, origin, dims), got), storage
        assert int((got != api.EMPTY).sum()) == s.info()["unique_voxels"]
        boxes[storage] = got
        s.close()
    assert np.array_equal(boxes["hashtable"], boxes["vcs"])


def config3_camera():
    """BASELINE.json config 3's view of the 512^3 terrain (tests/test_configs_gpu.py)."""
    return api.Camera((-96.0, 352.0, -96.0), (256.0, 64.0, 256.0), (0.0, 1.0, 0.0), 60.0, np.float32(3840) / np.float32(2160))


@pytest.fixture(scope="module")
def terrain_volume():
    """scenes.terrain(512, 1234) as a dense volume: vol[x, y, z] = colour(y) iff y < clip(h[x, z], 1, 511)."""
    h = np.clip(scenes.terrain_heights(512, 1234), 1, 511)
    y = np.arange(512, dtype=np.int32)
    colour = scenes._height_colour(y).astype(np.uint32)
    return np.where(y[None, :, None] < h[:, None, :], colour[None, :, None], np.uint32(api.EMPTY)).astype(np.uint32)


@pytest.mark.parametrize("storage", STORAGES)
def test_full_size_terrain(terrain_volume, storage):
    """BASELINE.json config 3: read_box of [0, 512)^3 (512 MB: more than one host slab) equals the host terrain; the same volume through
    add_dense_device renders config 3's 3840x2160 frame bit-identically to the list-built scene."""
    listed = api.VoxelScene(0)
    n = listed.generate_terrain(512, 1234)
    listed.generate_voxel_scene(storage)
    got = listed.read_box((0, 0, 0), (512, 512, 512))
    assert np.array_equal(got, terrain_volume)
    del got
    d_vol = to_device(terrain_volume)
    dense = api.VoxelScene(0)
    assert dense.add_dense_device(d_vol.data_ptr(), (512, 512, 512)) == n
    dense.generate_voxel_scene(storage)
    del d_vol
    assert dense.info() == listed.info()
    for algo in ("original", "longestaxis"):
        a = listed.render(3840, 2160, algo, config3_camera(), want_hits=True)
        b = dense.render(3840, 2160, algo, config3_camera(), want_hits=True)
        assert np.array_equal(a["hits"], b["hits"]) and np.array_equal(a["rgb"], b["rgb"]), (storage, algo)
        assert a["hits"][..., 3].mean() > 0.3


def test_errors_are_reported_before_any_device_work():
    import torch
    lib = api.load_library()
    i3 = lambda v: np.ascontiguousarray(np.asarray(v, np.int32))       # noqa: E731
    u3 = lambda v: np.ascontiguousarray(np.asarray(v, np.uint32))      # noqa: E731
    p = api._ptr
    n = C.c_uint64(123)
    vol = np.zeros((4, 4, 4), np.uint32)
    out = np.zeros(64, np.uint32)
    d_buf = torch.zeros(1024, dtype=torch.int32, device="cuda")
    misaligned = d_buf.data_ptr() + 2
    s = api.VoxelScene(0)
    # before build: read_box -> STATE
    assert lib.vrm_scene_read_box(s.h, p(i3((0, 0, 0))), p(u3((4, 4, 4))), p(out)) == 3
    assert lib.vrm_scene_read_box_device(s.h, p(i3((0, 0, 0))), p(u3((4, 4, 4))), C.c_void_p(d_buf.data_ptr())) == 3
    # coordinates out of range -> INVALID (|c| < 2^23 for every cell)
    for o, d in [((-(1 << 23), 0, 0), (4, 4, 4)), ((0, (1 << 23) - 3, 0), (4, 4, 4)), ((0, 0, 1 << 30), (1, 1, 1))]:
        assert lib.vrm_scene_add_dense(s.h, p(vol), p(u3(d)), p(i3(o)), api.EMPTY, C.byref(n)) == 1, o
        assert n.value == 0
    # misaligned device pointer -> INVALID
    assert lib.vrm_scene_add_dense_device(s.h, C.c_void_p(misaligned), p(u3((4, 4, 4))), p(i3((0, 0, 0))), 0, None) == 1
    # zero dims -> OK, nothing added
    for d in [(0, 4, 4), (4, 0, 4), (4, 4, 0)]:
        n.value = 123
        assert lib.vrm_scene_add_dense(s.h, p(vol), p(u3(d)), p(i3((0, 0, 0))), 0, C.byref(n)) == 0 and n.value == 0
        assert lib.vrm_scene_add_dense_device(s.h, C.c_void_p(misaligned), p(u3(d)), p(i3((0, 0, 0))), 0, None) == 0
    assert s.add_dense(np.zeros((0, 3, 3), np.uint32)) == 0
    s.generate_voxel_scene("vcs")
    assert s.info()["unique_voxels"] == 0
    # after build: add_dense -> STATE
    assert lib.vrm_scene_add_dense(s.h, p(vol), p(u3((4, 4, 4))), p(i3((0, 0, 0))), 0, C.byref(n)) == 3
    assert lib.vrm_scene_add_dense_device(s.h, C.c_void_p(d_buf.data_ptr()), p(u3((4, 4, 4))), p(i3((0, 0, 0))), 0, None) == 3
    # read_box: origin + dims overflowing int32 -> INVALID; misaligned device output -> INVALID; zero dims -> OK
    assert lib.vrm_scene_read_box(s.h, p(i3((0, 2**31 - 4, 0))), p(u3((1, 4, 1))), p(out)) == 1
    assert lib.vrm_scene_read_box_device(s.h, p(i3((0, 0, 0))), p(u3((4, 4, 4))), C.c_void_p(misaligned)) == 1
    assert lib.vrm_scene_read_box(s.h, p(i3((0, 0, 0))), p(u3((4, 0, 4))), p(out)) == 0
    with pytest.raises(api.VrmError):
        s.add_dense(vol)
    assert s.read_box((0, 2**31 - 5, 0), (1, 4, 1)).shape == (1, 4, 1)   # the largest legal end: origin + dims = INT32_MAX
    torch.cuda.synchronize()
