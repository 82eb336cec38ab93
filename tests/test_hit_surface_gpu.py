"""GPU tier (pytest -m gpu): vrm_hit_surface_* on the real kernel against the numpy restatement of the definition (tests/surface_ref.py),
bit for bit, on hit maps and traces the library itself produced."""
import os
import subprocess

import numpy as np
import pytest

import bench
from tests import surface_ref as sr
from tests.common import COMBOS, PROBE_CAMERAS, ROOT
from voxelraymarcher_b200 import api, scenes

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

W, H = 333, 187   # ragged: neither a multiple of the kernel's 4 records per thread nor of a warp
CLI = os.path.join(ROOT, "voxelraymarcher_b200", "VoxelRaymarcher")


def _scene(fill, storage):
    s = api.VoxelScene(0)
    fill(s)
    s.generate_voxel_scene(storage)
    return s


def _probe(s):
    s.add_voxels(*scenes.probe_scene())


def _cam(o, l, fov, w, h):
    return api.Camera(o, l, (0.0, 1.0, 0.0), fov, np.float32(w) / np.float32(h))


@pytest.fixture(scope="module")
def probe_scenes():
    out = {st: _scene(_probe, st) for st in ("hashtable", "vcs")}
    yield out
    for s in out.values():
        s.close()


@pytest.mark.parametrize("storage,algorithm", COMBOS)
@pytest.mark.parametrize("scale,translation", [(8, (0.0, 0.0, 0.0)), (8, (0.75, -1.25, 2.5)), (5, (-3.5, 0.25, 1.0))])
def test_probe_views(probe_scenes, storage, algorithm, scale, translation):
    s = probe_scenes[storage]
    cams = [_cam(o, l, fov, W, H) for o, l, fov in PROBE_CAMERAS]
    frames = [s.render(W, H, algorithm, c, scale=scale, translation=translation, want_hits=True, want_surface=True) for c in cams]
    hits = np.stack([f["hits"] for f in frames])
    assert hits[..., 3].sum() > 1000
    want_d, want_f = sr.views(hits, [c.data for c in cams], W, H, scale, translation)
    # render(want_surface=True) == render + hit_surface_views, one view at a time (camera in the kernel arguments) ...
    assert sr.same_bits(np.stack([f["depth"] for f in frames]), want_d)
    assert np.array_equal(np.stack([f["face"] for f in frames]), want_f)
    # ... and as a batch (cameras uploaded), host and device variants
    got_d, got_f = s.hit_surface_views(hits, cams, W, H, scale, translation)
    assert sr.same_bits(got_d, want_d) and np.array_equal(got_f, want_f)
    d_hits = torch.from_numpy(hits).cuda()
    d_depth = torch.empty((len(cams), H, W), dtype=torch.float32, device="cuda")
    d_face = torch.empty((len(cams), H, W), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    s.hit_surface_views_device(d_hits.data_ptr(), cams, W, H, d_depth.data_ptr(), d_face.data_ptr(), scale, translation)
    s.synchronize()
    assert sr.same_bits(d_depth.cpu().numpy(), want_d) and np.array_equal(d_face.cpu().numpy(), want_f)


def test_terrain_orbit_batch_device():
    """A render_views_device batch of bench orbit views of the 512^3 terrain, surfaces computed on the device from its hit map."""
    s = _scene(lambda sc: sc.generate_terrain(bench.SCENE_SIZE, bench.SCENE_SEED), "vcs")
    w, h = 1920, 1080
    cams = [bench.orbit_camera(api, v) for v in (0, 11, 22, 37, 50, 63)]
    n = len(cams)
    rgb = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
    hits = torch.empty((n, h, w, 4), dtype=torch.int32, device="cuda")
    depth = torch.empty((n, h, w), dtype=torch.float32, device="cuda")
    face = torch.empty((n, h, w), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    s.render_views_device(w, h, "longestaxis", cams, rgb.data_ptr(), hits.data_ptr())
    s.hit_surface_views_device(hits.data_ptr(), cams, w, h, depth.data_ptr(), face.data_ptr())
    s.synchronize()
    hits_h = hits.cpu().numpy()
    assert hits_h[..., 3].mean() > 0.1
    want_d, want_f = sr.views(hits_h, [c.data for c in cams], w, h)
    assert sr.same_bits(depth.cpu().numpy(), want_d)
    assert np.array_equal(face.cpu().numpy(), want_f)
    # only one output, and an output at an odd address (element-wise stores instead of vector stores)
    face2 = torch.zeros(n * h * w + 1, dtype=torch.uint8, device="cuda")
    s.hit_surface_views_device(hits.data_ptr(), cams, w, h, None, face2.data_ptr() + 1)
    s.synchronize()
    assert np.array_equal(face2[1:].cpu().numpy().reshape(n, h, w), want_f)
    s.close()


@pytest.fixture(scope="module")
def config5():
    s = _scene(lambda sc: sc.generate_sparse_shells(1024, 64, 11, 35), "vcs")
    yield s, scenes.random_rays(3840 * 2160, (512.0 + 31.5, 512.0 + 31.5, 512.0 + 31.5), seed=42)
    s.close()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("algorithm", ["longestaxis", "original"])
def test_config5_rays(config5, algorithm):
    """configs[4]'s incoherent rays, the full buffer: host (trace_rays(want_surface=True)) and device variants."""
    s, rays = config5
    got = s.trace_rays(rays, algorithm, want_hits=True, want_surface=True)
    assert got["hits"][:, 3].mean() > 0.2
    want_d, want_f = sr.rays(got["hits"], rays)
    assert sr.same_bits(got["depth"], want_d) and np.array_equal(got["face"], want_f)
    d_rays, d_hits = torch.from_numpy(rays).cuda(), torch.from_numpy(got["hits"]).cuda()
    d_depth = torch.empty(len(rays), dtype=torch.float32, device="cuda")
    d_face = torch.empty(len(rays), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    s.hit_surface_rays_device(d_hits.data_ptr(), d_rays.data_ptr(), len(rays), d_depth.data_ptr(), d_face.data_ptr())
    s.synchronize()
    assert sr.same_bits(d_depth.cpu().numpy(), want_d) and np.array_equal(d_face.cpu().numpy(), want_f)


@pytest.mark.parametrize("storage,algorithm", COMBOS)
def test_pixel_rays_traced_agree_with_render(probe_scenes, storage, algorithm):
    """The pixel rays of a frame traced as world rays: same hits, same faces, and render depth == len + trace depth exactly."""
    s = probe_scenes[storage]
    tr = (0.75, -1.25, 2.5)
    for o, l, fov in PROBE_CAMERAS:
        cam = _cam(o, l, fov, W, H)
        frame = s.render(W, H, algorithm, cam, scale=8, translation=tr, want_hits=True, want_surface=True)
        P, D, length = sr.pixel_rays(cam.data, W, H)
        rays = np.concatenate([P, D], -1).reshape(-1, 6)
        got = s.trace_rays(rays, algorithm, scale=8, translation=tr, want_hits=True, want_surface=True)
        assert np.array_equal(got["hits"], frame["hits"].reshape(-1, 4))
        assert np.array_equal(got["face"], frame["face"].reshape(-1))
        assert sr.same_bits((length.reshape(-1) + got["depth"]).astype(np.float32), frame["depth"].reshape(-1))


def test_all_miss_and_unbuilt_handle(probe_scenes):
    """A frame that hits nothing is +inf / 0 everywhere; the calls depend only on their arguments, so an unbuilt handle computes
    the same surfaces from a hit map."""
    s = probe_scenes["vcs"]
    cam = _cam((0.0, 40.0, 0.0), (0.0, 80.0, 1.0), 60.0, W, H)   # looking up, away from everything
    frame = s.render(W, H, "longestaxis", cam, scale=8, want_hits=True, want_surface=True)
    assert frame["hits"][..., 3].sum() == 0
    assert np.isposinf(frame["depth"]).all() and (frame["face"] == 0).all()
    rng = np.random.default_rng(3)
    hits = np.concatenate([rng.integers(-200, 200, (2, H, W, 3)), rng.integers(0, 2, (2, H, W, 1))], -1).astype(np.int32)
    cams = [_cam(o, l, fov, W, H) for o, l, fov in PROBE_CAMERAS[:2]]
    fresh = api.VoxelScene(0)
    got_d, got_f = fresh.hit_surface_views(hits, cams, W, H, 3, (1.0, 2.0, -0.5))
    want_d, want_f = sr.views(hits, [c.data for c in cams], W, H, 3, (1.0, 2.0, -0.5))
    assert sr.same_bits(got_d, want_d) and np.array_equal(got_f, want_f)
    fresh.close()


def test_argument_errors(probe_scenes):
    s = probe_scenes["vcs"]
    lib = s.lib
    cam = np.ascontiguousarray(_cam(*PROBE_CAMERAS[0], 64, 32).data)
    tr = np.zeros(3, np.float32)
    hits = torch.zeros(64 * 32 * 4 + 4, dtype=torch.int32, device="cuda")
    depth = torch.zeros(64 * 32 + 1, dtype=torch.float32, device="cuda")
    face = torch.zeros(64 * 32 + 4, dtype=torch.uint8, device="cuda")
    p = lambda a: a.ctypes.data  # noqa: E731
    views = lambda h, d, f, w=64, n=1: lib.vrm_hit_surface_views_device(s.h, p(cam), n, p(tr), 8, w, 32, h, d, f)  # noqa: E731
    assert views(hits.data_ptr(), depth.data_ptr(), face.data_ptr()) == 0
    assert views(hits.data_ptr() + 4, depth.data_ptr(), face.data_ptr()) == 1        # hits not 16-byte aligned
    assert views(hits.data_ptr(), depth.data_ptr() + 2, face.data_ptr()) == 1        # depth not 4-byte aligned
    assert views(hits.data_ptr(), None, None) == 1                                   # both outputs NULL
    assert views(hits.data_ptr(), depth.data_ptr() + 4, face.data_ptr() + 1) == 0    # 4-byte depth / any face alignment is legal
    assert views(hits.data_ptr(), depth.data_ptr(), None, w=0) == 0                   # zero records
    assert views(hits.data_ptr(), depth.data_ptr(), None, n=0) == 0
    rays = torch.zeros(64 * 6 + 1, dtype=torch.float32, device="cuda")
    assert lib.vrm_hit_surface_rays_device(s.h, rays.data_ptr(), 0, p(tr), 1, None, depth.data_ptr(), None) == 0   # n = 0
    assert lib.vrm_hit_surface_rays_device(s.h, rays.data_ptr(), 64, p(tr), 1, hits.data_ptr() + 8, depth.data_ptr(), None) == 1
    assert lib.vrm_hit_surface_rays_device(s.h, rays.data_ptr() + 2, 64, p(tr), 1, hits.data_ptr(), depth.data_ptr(), None) == 1
    assert lib.vrm_hit_surface_rays(s.h, None, 0, p(tr), 1, None, None, None) == 1                                    # both NULL
    assert lib.vrm_hit_surface_rays(None, None, 0, p(tr), 1, None, None, None) == 1
    s.synchronize()


def _read_pfm(path):
    with open(path, "rb") as f:
        assert f.readline() == b"Pf\n"
        w, h = (int(v) for v in f.readline().split())
        assert float(f.readline()) < 0     # little-endian
        data = np.frombuffer(f.read(), "<f4")
    assert data.size == w * h
    return data.reshape(h, w)[::-1]        # PFM rows run bottom to top


# the CLI reads its options only after all three positional arguments (cli/main.cpp)
@pytest.mark.parametrize("argv,storage,algo", [(["8", "hashtable", "original"], "hashtable", "original"), (["8", "vcs", "longestaxis"], "vcs", "longestaxis")])
def test_cli_depth_pfm(tmp_path, probe_scenes, argv, storage, algo):
    xyz, rgb = scenes.probe_scene()
    os.makedirs(tmp_path / "resources")
    scenes.write_csv(str(tmp_path / "resources" / "scene.vox"), xyz, rgb)
    p = subprocess.run([CLI, *argv, "--width", str(W), "--height", str(H), "--depth", "depth.pfm"], stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, cwd=tmp_path)
    assert p.returncode == 0, p.stdout
    assert "ERROR" not in p.stdout
    got = _read_pfm(tmp_path / "depth.pfm")
    want = probe_scenes[storage].render(W, H, algo, api.Camera.reference_default(W, H), scale=8, want_surface=True)["depth"]
    assert sr.same_bits(np.ascontiguousarray(got), want)
    assert np.isposinf(got).any() and np.isfinite(got).any()
