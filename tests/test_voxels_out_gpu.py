"""GPU tier: the stored voxels of a built scene as a voxel list, box by box, in C order (vrm_scene_read_voxels[_device]).

read_voxels(origin, dims) must be the non-EMPTY cells of read_box(origin, dims) in linear-index order -- coordinates and colours bit
for bit -- for both storage types, on boxes that start and end inside clusters, cross region and region-table edges or lie outside the
table.  Whole scenes are checked against a last-wins dedupe of the staged list, by rebuilding and rendering, and at full size (512^3
terrain, 2048^3 sparse shells with 64-bit sort keys) by order + lookup + count, without a dense oracle."""
import ctypes as C

import numpy as np
import pytest

from tests.common import PROBE_CAMERAS, scenes
from tests.test_dense_gpu import VOL_ORIGIN, VOL_SHAPE, random_volume
from voxelraymarcher_b200 import api

pytestmark = pytest.mark.gpu

STORAGES = ["hashtable", "vcs"]


def expected_from_box(vol, origin):
    """read_box output without the empties, as the voxel list read_voxels must return."""
    mask = vol != api.EMPTY
    return (np.argwhere(mask) + np.asarray(origin, np.int64)).astype(np.int32), vol[mask].astype(np.uint32)


def built(xyz, rgb, storage):
    s = api.VoxelScene(0)
    s.add_voxels(xyz, rgb)
    s.generate_voxel_scene(storage)
    return s


def check_box(s, origin, dims):
    want_xyz, want_rgb = expected_from_box(s.read_box(origin, dims), origin)
    xyz, rgb = s.read_voxels(origin, dims)
    assert xyz.dtype == np.int32 and rgb.dtype == np.uint32 and xyz.shape == (len(rgb), 3)
    assert np.array_equal(xyz, want_xyz), (origin, dims, len(xyz), len(want_xyz))
    assert np.array_equal(rgb, want_rgb), (origin, dims)
    assert s.count_voxels(origin, dims) == len(want_rgb)
    return len(want_rgb)


def boxes_for(s, seed):
    """Boxes of every kind the contract names, relative to the scene's region table."""
    (o, d) = [np.asarray(v, np.int64) for v in s.scene_box()]
    rng = np.random.default_rng(seed)
    out = [(o, d),                                       # the whole scene_box
           (o + 3, d - 9),                               # starts and ends inside clusters on every axis
           (o - 37, d + 70),                             # crosses the region-table edges on every side
           (o + d + 5, np.array([9, 4, 30])),            # wholly outside the table
           (o - 100, np.array([40, 700, 3]))]            # outside on x, crossing on y and z
    for a in range(3):                                   # one cell thick along each axis, in the middle of a cluster
        lo, dd = o + 5, d - 13
        lo[a] = o[a] + d[a] // 2 + 3
        dd[a] = 1
        out.append((lo, dd))
    for _ in range(6):                                   # random boxes crossing region edges (64) and cluster edges (8)
        lo = o + rng.integers(-20, d)
        out.append((lo, rng.integers(1, np.minimum(d, 150) + 1)))
    return [(tuple(int(v) for v in a), tuple(int(v) for v in b)) for a, b in out]


def scene_voxels(name):
    if name == "volume":
        vol = random_volume(VOL_SHAPE, seed=2024)
        mask = vol != api.EMPTY
        return (np.argwhere(mask) + np.asarray(VOL_ORIGIN)).astype(np.int32), vol[mask]
    return scenes.probe_scene() if name == "probe" else scenes.mini_scene()


@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("name", ["volume", "probe", "mini"])
def test_equals_read_box_without_empties(name, storage):
    xyz, rgb = scene_voxels(name)
    s = built(xyz, rgb, storage)
    total = 0
    for origin, dims in boxes_for(s, seed=len(name)):
        total += check_box(s, origin, dims)
    assert total > 0
    # single cells: stored voxels, empty cells, cells outside the table
    picks = np.concatenate([xyz[:: max(1, len(xyz) // 25)], np.array([[0, 0, 0], [-1, -1, -1], [5000, 0, 0], [-129, 3, 100]], np.int32)])
    for p in picks:
        check_box(s, tuple(int(v) for v in p), (1, 1, 1))
    assert s.count_voxels() == s.info()["unique_voxels"]


def test_mini_scene_contents_and_storage_independence():
    """The staged mini scene has duplicates with different colours: both storage types list exactly the last-wins dedupe, sorted."""
    xyz, rgb = scenes.mini_scene()
    last = {}
    for p, c in zip(map(tuple, xyz.tolist()), rgb.tolist()):
        last[p] = c
    keys = sorted(last)
    want_xyz = np.array(keys, np.int32)
    want_rgb = np.array([last[k] for k in keys], np.uint32)
    assert len(keys) < len(xyz)
    lists = {}
    for storage in STORAGES:
        s = built(xyz, rgb, storage)
        got_xyz, got_rgb = s.read_voxels()
        assert len(got_rgb) == s.info()["unique_voxels"] == len(keys)
        assert np.array_equal(got_xyz, want_xyz) and np.array_equal(got_rgb, want_rgb), storage
        lists[storage] = (got_xyz, got_rgb)
    # the same holds for a box of the probe scene cut through several regions
    pxyz, prgb = scenes.probe_scene()
    for storage in STORAGES:
        s = built(pxyz, prgb, storage)
        lists[storage + "_probe"] = s.read_voxels((-77, -3, -60), (190, 70, 150))
    assert np.array_equal(lists["hashtable_probe"][0], lists["vcs_probe"][0])
    assert np.array_equal(lists["hashtable_probe"][1], lists["vcs_probe"][1])


@pytest.mark.parametrize("storage", STORAGES)
def test_round_trip_renders_identically(storage):
    xyz, rgb = scenes.probe_scene()
    s = built(xyz, rgb, storage)
    lx, lrgb = s.read_voxels()
    r = built(lx, lrgb, storage)
    assert r.info() == s.info()
    w, h = 320, 180
    for algo in ("original", "longestaxis"):
        for o, look, fov in PROBE_CAMERAS:
            cam = api.Camera(o, look, (0.0, 1.0, 0.0), fov, np.float32(w) / np.float32(h))
            a = s.render(w, h, algo, cam, scale=8, want_hits=True)
            b = r.render(w, h, algo, cam, scale=8, want_hits=True)
            assert np.array_equal(a["hits"], b["hits"]) and np.array_equal(a["rgb"], b["rgb"]), (storage, algo, o)
    # and the other storage type, built from the list, holds the same voxels
    other = built(lx, lrgb, "vcs" if storage == "hashtable" else "hashtable")
    ox, orgb = other.read_voxels()
    assert np.array_equal(ox, lx) and np.array_equal(orgb, lrgb)


@pytest.mark.parametrize("storage", STORAGES)
def test_colour_equal_to_empty_is_listed(storage):
    xyz = np.array([[1, 2, 3], [1, 2, 4], [70, -5, 9], [-3, 0, 0]], np.int32)
    rgb = np.array([0x123456, api.EMPTY, api.EMPTY, 7], np.uint32)
    s = built(xyz, rgb, storage)
    got_xyz, got_rgb = s.read_voxels()
    order = np.lexsort((xyz[:, 2], xyz[:, 1], xyz[:, 0]))
    assert np.array_equal(got_xyz, xyz[order]) and np.array_equal(got_rgb, rgb[order])
    assert s.count_voxels() == s.info()["unique_voxels"] == 4
    # read_box cannot tell those two cells from empty ones: the documented single difference
    box_xyz, _ = expected_from_box(s.read_box(*s.scene_box()), s.scene_box()[0])
    assert len(box_xyz) == 2


def read_voxels_device(s, origin, dims, capacity=None):
    import torch
    n = s.count_voxels(origin, dims)
    cap = n if capacity is None else capacity
    d_xyz = torch.full((max(cap, 1), 3), -7, dtype=torch.int32, device="cuda")
    d_rgb = torch.full((max(cap, 1),), -7, dtype=torch.int32, device="cuda")
    got = s.read_voxels_device(origin, dims, d_xyz.data_ptr(), d_rgb.data_ptr(), cap)
    assert got == n
    s.synchronize()
    return d_xyz[:n].cpu().numpy(), d_rgb[:n].cpu().numpy().view(np.uint32)


def is_c_order(xyz):
    k = xyz.astype(np.int64) + (1 << 20)
    key = (k[:, 0] << 42) | (k[:, 1] << 21) | k[:, 2]
    return bool((np.diff(key) > 0).all())


@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("scene", ["terrain512", "shells2048"])
def test_full_size(scene, storage):
    """BASELINE.json configs[3]-sized scenes: the whole-scene list is strictly increasing in (x, y, z), every listed coordinate looks up
    to the listed colour and the length is unique_voxels -- together: exactly the stored set in C order.  The 2048^3 scene (33 key
    bits) takes the 64-bit sort."""
    s = api.VoxelScene(0)
    if scene == "terrain512":
        s.generate_terrain(512, 1234)
    else:
        s.generate_sparse_shells(2048, 64, 7, 35)
    s.generate_voxel_scene(storage)
    info = s.info()
    origin, dims = s.scene_box()
    xyz, rgb = read_voxels_device(s, origin, dims)
    assert len(rgb) == info["unique_voxels"] > 10_000_000
    assert is_c_order(xyz)
    assert np.array_equal(s.lookup(xyz)[0], rgb)
    hx, hrgb = s.read_voxels()
    assert np.array_equal(hx, xyz) and np.array_equal(hrgb, rgb)
    del hx, hrgb, xyz, rgb
    if scene == "shells2048":
        sub = ((517, 259, 1031), (512, 512, 512))
        n = check_box(s, *sub)
        assert n > 100_000


@pytest.mark.parametrize("storage", STORAGES)
def test_host_and_device_agree(storage):
    xyz, rgb = scene_voxels("volume")
    s = built(xyz, rgb, storage)
    for origin, dims in boxes_for(s, seed=5)[:8]:
        hx, hrgb = s.read_voxels(origin, dims)
        dx, drgb = read_voxels_device(s, origin, dims)
        assert np.array_equal(hx, dx) and np.array_equal(hrgb, drgb), (origin, dims)
        # a larger buffer than needed is fine: the count is returned, the rest is left alone
        dx2, drgb2 = read_voxels_device(s, origin, dims, capacity=len(hrgb) + 100)
        assert np.array_equal(hx, dx2) and np.array_equal(hrgb, drgb2)
    # count only, both variants
    lib = api.load_library()
    o, d = api._box(*s.scene_box())
    n = C.c_uint64(5)
    assert lib.vrm_scene_read_voxels(s.h, api._ptr(o), api._ptr(d), None, None, 0, C.byref(n)) == 0 and n.value == len(xyz)
    n.value = 5
    assert lib.vrm_scene_read_voxels_device(s.h, api._ptr(o), api._ptr(d), None, None, 0, C.byref(n)) == 0 and n.value == len(xyz)


def test_status_codes():
    import torch
    lib = api.load_library()
    i3 = lambda v: np.ascontiguousarray(np.asarray(v, np.int32))       # noqa: E731
    u3 = lambda v: np.ascontiguousarray(np.asarray(v, np.uint32))      # noqa: E731
    p = api._ptr
    xyz, rgb = scene_voxels("mini")
    s = api.VoxelScene(0)
    s.add_voxels(xyz, rgb)
    o, d = i3((-128, -128, -128)), u3((256, 256, 256))   # the mini scene's scene_box
    n = C.c_uint64(123)
    hx = np.zeros((4, 3), np.int32)
    hr = np.zeros(4, np.uint32)
    d_buf = torch.zeros(4096, dtype=torch.int32, device="cuda")
    # before build: STATE
    assert lib.vrm_scene_read_voxels(s.h, p(o), p(d), p(hx), p(hr), 4, C.byref(n)) == 3 and n.value == 0
    assert lib.vrm_scene_read_voxels_device(s.h, p(o), p(d), C.c_void_p(d_buf.data_ptr()), C.c_void_p(d_buf.data_ptr() + 4096), 4, C.byref(n)) == 3
    s.generate_voxel_scene("vcs")
    assert s.scene_box() == ((-128,) * 3, (256,) * 3)
    count = s.info()["unique_voxels"]
    # n_out is required
    assert lib.vrm_scene_read_voxels(s.h, p(o), p(d), None, None, 0, None) == 1
    # origin + dims overflowing int32: INVALID
    assert lib.vrm_scene_read_voxels(s.h, p(i3((0, 2**31 - 4, 0))), p(u3((1, 4, 1))), None, None, 0, C.byref(n)) == 1
    assert lib.vrm_scene_read_voxels(s.h, p(i3((0, 2**31 - 5, 0))), p(u3((1, 4, 1))), None, None, 0, C.byref(n)) == 0 and n.value == 0
    # exactly one output NULL: INVALID
    assert lib.vrm_scene_read_voxels(s.h, p(o), p(d), p(hx), None, 4, C.byref(n)) == 1
    assert lib.vrm_scene_read_voxels(s.h, p(o), p(d), None, p(hr), 4, C.byref(n)) == 1
    assert lib.vrm_scene_read_voxels_device(s.h, p(o), p(d), C.c_void_p(d_buf.data_ptr()), None, 4, C.byref(n)) == 1
    # capacity one short: INVALID, n_out holds the count, the buffers are untouched
    sx = np.full((count, 3), -5, np.int32)
    sr = np.full(count, 0xDEADBEEF, np.uint32)
    n.value = 0
    assert lib.vrm_scene_read_voxels(s.h, p(o), p(d), p(sx), p(sr), count - 1, C.byref(n)) == 1 and n.value == count
    assert (sx == -5).all() and (sr == 0xDEADBEEF).all()
    t_xyz = torch.full((count, 3), -5, dtype=torch.int32, device="cuda")
    t_rgb = torch.full((count,), -5, dtype=torch.int32, device="cuda")
    n.value = 0
    assert lib.vrm_scene_read_voxels_device(s.h, p(o), p(d), C.c_void_p(t_xyz.data_ptr()), C.c_void_p(t_rgb.data_ptr()), count - 1, C.byref(n)) == 1
    assert n.value == count
    s.synchronize()
    assert (t_xyz == -5).all().item() and (t_rgb == -5).all().item()
    # the same buffers with the full capacity: OK
    assert lib.vrm_scene_read_voxels(s.h, p(o), p(d), p(sx), p(sr), count, C.byref(n)) == 0 and n.value == count
    assert np.array_equal(sx, s.read_voxels()[0])
    # misaligned device pointers: INVALID
    base = d_buf.data_ptr()
    assert lib.vrm_scene_read_voxels_device(s.h, p(o), p(d), C.c_void_p(base + 2), C.c_void_p(base + 8192), 1000, C.byref(n)) == 1
    assert lib.vrm_scene_read_voxels_device(s.h, p(o), p(d), C.c_void_p(base), C.c_void_p(base + 8193), 1000, C.byref(n)) == 1
    # zero dims: OK and 0
    for z in [(0, 4, 4), (4, 0, 4), (4, 4, 0)]:
        n.value = 123
        assert lib.vrm_scene_read_voxels(s.h, p(o), p(u3(z)), p(hx), p(hr), 4, C.byref(n)) == 0 and n.value == 0
        n.value = 123
        assert lib.vrm_scene_read_voxels_device(s.h, p(o), p(u3(z)), C.c_void_p(base), C.c_void_p(base + 8192), 4, C.byref(n)) == 0
        assert n.value == 0
    assert s.count_voxels((0, 0, 0), (0, 5, 5)) == 0
    # an empty built scene lists nothing
    e = api.VoxelScene(0)
    e.generate_voxel_scene("hashtable")
    assert e.count_voxels() == 0 and e.read_voxels()[0].shape == (0, 3)
    torch.cuda.synchronize()
