"""GPU tier (pytest -m gpu): vrm_cast_* on the real kernel against the numpy cell-by-cell walk of tests/cast_ref.py, bit for bit, on the
inputs of the CPU tier and on the bench scenes, plus the kernel's self-consistency with the hit surfaces and its argument checks."""
import numpy as np
import pytest

import bench
from tests import cast_ref as cr
from tests import surface_ref as sr
from tests.common import MINI_CAMERAS, PROBE_CAMERAS
from tests.test_cast import SCENES
from voxelraymarcher_b200 import api, scenes

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

W, H = 96, 54
_CACHE = {}


def _cam(o, l, fov, w, h):
    return api.Camera(o, l, (0.0, 1.0, 0.0), fov, np.float32(w) / np.float32(h))


def built(name, storage):
    """(Stored, VoxelScene, scale, translation) of a CPU-tier scene."""
    key = (name, storage)
    if key not in _CACHE:
        fn, scale, tr = SCENES[name]
        xyz, rgb = fn()
        s = api.VoxelScene(0)
        s.add_voxels(xyz, rgb)
        s.generate_voxel_scene(storage)
        _CACHE[key] = (cr.Stored(xyz, rgb), s, scale, tr)
    return _CACHE[key]


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("storage", ["vcs", "hashtable"])
@pytest.mark.parametrize("name", list(SCENES))
def test_rays_match_numpy_walk(name, storage):
    st, s, scale, tr = built(name, storage)
    cases = cr.ray_cases(st, scale, tr, seed=len(name), n=800 if name in ("terrain192", "shells512") else 1500)
    for case, rays in cases.items():
        for rname, ranges in cr.range_cases(len(rays)).items():
            if case not in ("random", "ties") and rname not in ("default", "interval"):
                continue
            got = s.cast_rays(rays, ranges, scale, tr)
            assert cr.same(got, cr.cast_rays(st, rays, ranges, scale, tr)), (case, rname)


@pytest.mark.parametrize("storage", ["vcs", "hashtable"])
@pytest.mark.parametrize("name", ["probe", "probe_translated", "mini"])
def test_views_match_numpy_walk(name, storage):
    st, s, scale, tr = built(name, storage)
    cams = [_cam(o, l, fov, W, H) for o, l, fov in (PROBE_CAMERAS if name.startswith("probe") else MINI_CAMERAS)]
    want = cr.cast_views(st, [c.data for c in cams], W, H, scale, tr)
    assert cr.same(s.cast_views(cams, W, H, scale, tr), want)           # batch: cameras uploaded
    one = s.cast_views(cams[:1], W, H, scale, tr)                        # one view: camera in the kernel arguments
    assert cr.same(one, {k: v[:1] for k, v in want.items()})


def _device_outputs(n, shape=()):
    return dict(hits=torch.empty((n, *shape, 4), dtype=torch.int32, device="cuda"), depth=torch.empty((n, *shape), dtype=torch.float32, device="cuda"),
                face=torch.empty((n, *shape), dtype=torch.uint8, device="cuda"), colour=torch.empty((n, *shape), dtype=torch.int32, device="cuda"))


def _host(out):
    h = {k: v.cpu().numpy() for k, v in out.items()}
    h["colour"] = h["colour"].view(np.uint32)
    return h


def test_host_equals_device_and_output_subsets():
    st, s, scale, tr = built("probe_translated", "hashtable")
    rays = cr.ray_cases(st, scale, tr, seed=4)["random"]
    ranges = cr.range_cases(len(rays))["interval"]
    want = s.cast_rays(rays, ranges, scale, tr)
    d_rays, d_ranges = torch.from_numpy(rays).cuda(), torch.from_numpy(ranges).cuda()
    full = _device_outputs(len(rays))
    torch.cuda.synchronize()
    s.cast_rays_device(d_rays.data_ptr(), len(rays), d_ranges.data_ptr(), *(full[k].data_ptr() for k in ("hits", "depth", "face", "colour")),
                       scale=scale, translation=tr)
    s.synchronize()
    assert cr.same(_host(full), want)
    keys = ("hits", "depth", "face", "colour")
    for mask in range(1, 16):
        part = _device_outputs(len(rays))
        for v in part.values():
            v.zero_()
        ptrs = [part[k].data_ptr() if mask >> i & 1 else None for i, k in enumerate(keys)]
        torch.cuda.synchronize()
        s.cast_rays_device(d_rays.data_ptr(), len(rays), d_ranges.data_ptr(), *ptrs, scale=scale, translation=tr)
        s.synchronize()
        h = _host(part)
        for i, k in enumerate(keys):
            if mask >> i & 1:
                assert np.array_equal(h[k].view(np.uint8), np.ascontiguousarray(want[k]).view(np.uint8)), (mask, k)
    # host subsets through the C ABI, and the views' device variant
    lib, p = s.lib, (lambda a: a.ctypes.data)
    depth = np.zeros(len(rays), np.float32)
    assert lib.vrm_cast_rays(s.h, p(rays), p(ranges), len(rays), p(np.asarray(tr, np.float32)), scale, None, p(depth), None, None) == 0
    assert sr.same_bits(depth, want["depth"])
    cams = [_cam(o, l, fov, W, H) for o, l, fov in PROBE_CAMERAS]
    vw = s.cast_views(cams, W, H, scale, tr)
    dv = _device_outputs(len(cams), (H, W))
    torch.cuda.synchronize()
    s.cast_views_device(cams, W, H, *(dv[k].data_ptr() for k in keys), scale=scale, translation=tr)
    s.synchronize()
    assert cr.same(_host(dv), vw)


def test_definition_edges_on_device():
    """A voxel stored with the colour EMPTY is hit; zero directions, start-cell hits and always-miss rays."""
    xyz = np.array([[2, 3, 4], [10, 3, 4]], np.int32)
    rgb = np.array([cr.EMPTY, 0x123456], np.uint32)
    st = cr.Stored(xyz, rgb)
    rays = np.array([[2.5, 3.5, 4.5, 0, 0, 0], [5.5, 3.5, 4.5, 0, 0, 0], [0.5, 3.5, 4.5, 1, 0, 0], [12.5, 3.5, 4.5, -2, 0, 0],
                     [0.5, 3.5, 4.5, -0.0, 0, 0], [np.nan, 3.5, 4.5, 1, 0, 0], [0.5, 3.5, 4.5, np.inf, 0, 0]], np.float32)
    ranges = np.array([[0.25, 1], [0, np.inf], [0, np.inf], [0, np.inf], [0, np.inf], [0, np.inf], [0, np.inf]], np.float32)
    for storage in ("vcs", "hashtable"):
        s = api.VoxelScene(0)
        s.add_voxels(xyz, rgb)
        s.generate_voxel_scene(storage)
        got = s.cast_rays(rays, ranges)
        assert cr.same(got, cr.cast_rays(st, rays, ranges))
        assert got["hits"][0].tolist() == [2, 3, 4, 1] and got["colour"][0] == cr.EMPTY and got["depth"][0] == np.float32(0.25)
        assert got["hits"][3].tolist() == [10, 3, 4, 1] and got["colour"][3] == 0x123456
        s.close()


def test_status_codes():
    lib = api.load_library()
    tr = np.zeros(3, np.float32)
    p = lambda a: a.ctypes.data  # noqa: E731
    rays = np.zeros((4, 6), np.float32)
    depth = np.zeros(4, np.float32)
    fresh = api.VoxelScene(0)
    assert lib.vrm_cast_rays(fresh.h, p(rays), None, 4, p(tr), 1, None, p(depth), None, None) == 3            # unbuilt: VRM_ERR_STATE
    assert lib.vrm_cast_views(fresh.h, p(np.zeros(15, np.float32)), 1, p(tr), 1, 4, 4, None, p(depth), None, None) == 3
    fresh.close()
    _, s, _, _ = built("mini", "vcs")
    assert lib.vrm_cast_rays(s.h, p(rays), None, 4, p(tr), 1, None, None, None, None) == 1                     # every output NULL
    assert lib.vrm_cast_rays(s.h, p(rays), None, 0, p(tr), 1, None, p(depth), None, None) == 0                 # n = 0
    assert lib.vrm_cast_rays(s.h, p(rays), None, 4, p(tr), 0, None, p(depth), None, None) == 1                 # scale 0
    assert lib.vrm_cast_rays(None, p(rays), None, 4, p(tr), 1, None, p(depth), None, None) == 1
    d_rays = torch.zeros(4 * 6 + 1, dtype=torch.float32, device="cuda")
    d_hits = torch.zeros(4 * 4 + 4, dtype=torch.int32, device="cuda")
    d_f = torch.zeros(8, dtype=torch.float32, device="cuda")
    rd = lambda r, g, h, dep, c: lib.vrm_cast_rays_device(s.h, r, g, 4, p(tr), 1, h, dep, None, c)  # noqa: E731
    assert rd(d_rays.data_ptr(), None, d_hits.data_ptr(), d_f.data_ptr(), None) == 0
    assert rd(d_rays.data_ptr(), None, d_hits.data_ptr() + 4, None, None) == 1                                 # hits not 16-byte aligned
    assert rd(d_rays.data_ptr() + 2, None, d_hits.data_ptr(), None, None) == 1                                 # rays not 4-byte aligned
    assert rd(d_rays.data_ptr(), d_f.data_ptr() + 2, d_hits.data_ptr(), None, None) == 1                       # ranges not 4-byte aligned
    assert rd(d_rays.data_ptr(), None, None, d_f.data_ptr() + 2, None) == 1                                    # depth not 4-byte aligned
    assert rd(d_rays.data_ptr(), None, None, None, d_f.data_ptr() + 2) == 1                                    # colour not 4-byte aligned
    assert rd(d_rays.data_ptr(), None, None, None, None) == 1                                                  # every output NULL
    cam = np.ascontiguousarray(_cam(*MINI_CAMERAS[0], 8, 8).data)
    assert lib.vrm_cast_views_device(s.h, p(cam), 1, p(tr), 1, 0, 8, None, d_f.data_ptr(), None, None) == 0    # zero records
    assert lib.vrm_cast_views_device(s.h, p(cam), 1, p(tr), 1, 8, 8, d_hits.data_ptr() + 4, None, None, None) == 1
    s.synchronize()


def test_terrain_bench_view_4k():
    """Every pixel's depth equals the hit surface of the cast's own hit map; a seeded 200 k-pixel sample equals the numpy walk."""
    xyz, rgb = scenes.terrain(bench.SCENE_SIZE, bench.SCENE_SEED)
    st = cr.Stored(xyz, rgb)
    s = api.VoxelScene(0)
    s.generate_terrain(bench.SCENE_SIZE, bench.SCENE_SEED)
    s.generate_voxel_scene("vcs")
    w, h = bench.WIDTH, bench.HEIGHT
    cam = bench.orbit_camera(api, 0)
    out = _device_outputs(1, (h, w))
    depth2 = torch.empty((1, h, w), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    s.cast_views_device([cam], w, h, *(out[k].data_ptr() for k in ("hits", "depth", "face", "colour")))
    s.hit_surface_views_device(out["hits"].data_ptr(), [cam], w, h, depth2.data_ptr(), None)
    s.synchronize()
    got = _host(out)
    assert got["hits"][..., 3].mean() > 0.1
    entered = (got["hits"][..., 3] != 0) & (got["face"] != 0)
    assert sr.same_bits(got["depth"][entered], depth2.cpu().numpy()[entered])
    pix = np.sort(np.random.default_rng(7).choice(w * h, 200_000, replace=False))
    want = cr.cast_pixels(st, cam.data, w, h, pix)
    assert cr.same({k: v.reshape(w * h, *v.shape[3:])[pix] for k, v in got.items()}, want)
    s.close()


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("storage", ["vcs", "hashtable"])
def test_config5_rays(storage):
    """configs[4]'s incoherent rays, the full buffer: depth equals the hit surface of the cast's own hits; a 200 k-ray sample equals numpy."""
    xyz, rgb = scenes.sparse_shells(1024, 64, 11, 35)
    s = api.VoxelScene(0)
    s.generate_sparse_shells(1024, 64, 11, 35)
    s.generate_voxel_scene(storage)
    rays = scenes.random_rays(3840 * 2160, (512.0 + 31.5,) * 3, seed=42)
    n = len(rays)
    d_rays = torch.from_numpy(rays).cuda()
    out = _device_outputs(n)
    depth2 = torch.empty(n, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    s.cast_rays_device(d_rays.data_ptr(), n, None, *(out[k].data_ptr() for k in ("hits", "depth", "face", "colour")))
    s.hit_surface_rays_device(out["hits"].data_ptr(), d_rays.data_ptr(), n, depth2.data_ptr(), None)
    s.synchronize()
    got = _host(out)
    assert got["hits"][:, 3].mean() > 0.2
    entered = (got["hits"][:, 3] != 0) & (got["face"] != 0)
    assert np.array_equal(got["depth"][entered], depth2.cpu().numpy()[entered])
    idx = np.sort(np.random.default_rng(11).choice(n, 200_000, replace=False))
    want = cr.cast_rays(cr.Stored(xyz, rgb), rays[idx])
    assert cr.same({k: v[idx] for k, v in got.items()}, want)
    s.close()
