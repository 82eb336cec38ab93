"""GPU tier: every BASELINE.json configuration at ITS OWN SIZE against the reference (VERDICT r01 row h).

The checker is the unmodified reference's host build (`refh`, all host cores: a 4K frame of the 512^3 terrain takes a second or
two) where oracle/Makefile has built it from a reference checkout, else its C restatement (`orc`,
oracle/vrm_oracle.c, which tests/test_oracle.py pins to the reference through the committed golden fixtures); for the 2048^3
orbit, where the reference crawls for seconds per frame, the reference's own CUDA kernels built with -fmad=false (`refgx`, same
IEEE arithmetic as the host build) where present, else the restatement as well.  Bar: bit-exact hit maps and RGB, and equal
event counters where the checker counts them (the host builds).  In addition every frame and ray buffer must equal, at the
seeded sample positions of tests.common.config_sample, the stored results in tests/golden/config_golden.npz, so that the
full-size outputs stay pinned even where no reference build is present and whichever checker runs.  Reference entry points:
main/Main.cu:195-199 (frame size, camera), renderer/Renderer.cuh:1033-1063 (kernels), :917-1010 / :338-434 (per-ray routines
used by config 5)."""
import os

import numpy as np
import pytest

from tests.common import COMBOS, GOLDEN_DIR, PROBE_CAMERAS, build_oracle, config_sample, oracle_kind, po, scenes
from voxelraymarcher_b200 import api

pytestmark = pytest.mark.gpu

CORES = os.cpu_count() or 1
CONFIG4_VIEWS = [3, 19, 38, 54]


def config3_camera():
    return api.Camera((-96.0, 352.0, -96.0), (256.0, 64.0, 256.0), (0.0, 1.0, 0.0), 60.0, np.float32(3840) / np.float32(2160))


def config5_rays():
    return scenes.random_rays(3840 * 2160, (512.0 + 31.5, 512.0 + 31.5, 512.0 + 31.5), seed=42)


@pytest.fixture(scope="module")
def golden():
    """tests/golden/config_golden.npz (tests/golden/make_golden.py configs): every frame and ray buffer of this module at the
    seeded positions of tests.common.config_sample, as the checker named in its `checker` entry computed them."""
    return np.load(os.path.join(GOLDEN_DIR, "config_golden.npz"))


def _check_golden(golden, key, hits, rgb=None, colour=None, counters=None):
    idx = config_sample(hits.size // 4)
    assert np.array_equal(hits.reshape(-1, 4)[idx], golden[f"{key}_hits"]), (key, "hit records differ from the stored sample")
    if rgb is not None:
        assert np.array_equal(rgb.reshape(-1, 3)[idx], golden[f"{key}_rgb"]), (key, "RGB differs from the stored sample")
    if colour is not None:
        assert np.array_equal(colour[idx], golden[f"{key}_colour"]), (key, "colours differ from the stored sample")
    if counters is not None:
        assert counters == golden[f"{key}_counters"].tolist(), (key, "event counters differ from the stored ones")


def _product(xyz, rgb, storage):
    s = api.VoxelScene(0)
    s.add_voxels(xyz, rgb)
    s.generate_voxel_scene(storage)
    return s


def _compare_frame(s, ref, cam, w, h, algo, scale, golden, key, counters=True, tag=""):
    s.set_statistics(counters)
    got = s.render(w, h, algo, cam, scale=scale, want_hits=True)
    st = s.get_statistics() if counters else None
    want = ref.render(cam.data, w, h, algo, scale=scale, want_counters=counters, threads=CORES)
    nbad = int((got["hits"] != want["hits"]).any(-1).sum())
    assert nbad == 0, (tag, algo, f"{nbad} hit-map pixels differ")
    assert np.array_equal(got["rgb"], want["rgb"]), (tag, algo, int((got["rgb"] != want["rgb"]).any(-1).sum()))
    mine = [st["exist_checks"], st["exist_false"], st["lookups"], st["lookup_hits"]] if counters else None
    if counters:
        assert mine == [int(v) for v in want["counters"][:4]], (tag, algo)
        assert st["rays"] == w * h
    _check_golden(golden, key, got["hits"], rgb=got["rgb"], counters=mine)
    return want


@pytest.fixture(scope="module")
def probe():
    return scenes.probe_scene()


def test_config1_scene_standin_hashtable_original_720p(probe, golden):
    """configs[0]: resources/scene.vox (stand-in, SURVEY.md F3), hashtable + original, 1280x720, the reference's camera and scale 8."""
    kind = oracle_kind()
    xyz, rgb = probe
    po.set_lighting(kind)
    s, ref = _product(xyz, rgb, "hashtable"), build_oracle(kind, xyz, rgb, "hashtable")
    cam = api.Camera.reference_default(1280, 720)
    want = _compare_frame(s, ref, cam, 1280, 720, "original", 8, golden, "config1_hashtable_original", tag="config1")
    assert int(want["hits"][..., 3].sum()) > 300_000
    s.close(); ref.close()


@pytest.mark.parametrize("storage", ["hashtable", "vcs"])
def test_config2_scene_standin_all_combos_1080p(probe, golden, storage):
    """configs[1]: the reference's native frame (1920x1080, Main.cu:195-199), all four storage x algorithm combinations, each against
    the same combination of the reference: host build (bit-exact, counters), -fmad=false CUDA build (bit-exact), default CUDA build
    (>= 99.9 % of the pixels within 1 LSB per channel, BASELINE.json north_star)."""
    kind = oracle_kind()
    xyz, rgb = probe
    po.set_lighting(kind)
    s, ref = _product(xyz, rgb, storage), build_oracle(kind, xyz, rgb, storage)
    cam = api.Camera.reference_default(1920, 1080)
    frames = {}
    for algo in ("original", "longestaxis"):
        _compare_frame(s, ref, cam, 1920, 1080, algo, 8, golden, f"config2_{storage}_{algo}", tag=f"config2 {storage}")
        frames[algo] = s.render(1920, 1080, algo, cam, scale=8, want_hits=True)
    ref.close()
    if po.available("refgx") and po.available("refg"):
        for kind in ("refgx", "refg"):
            po.set_lighting(kind)
            g = build_oracle(kind, xyz, rgb, storage)
            for algo in ("original", "longestaxis"):
                want = g.render(cam.data, 1920, 1080, algo, scale=8)
                if kind == "refgx":
                    assert np.array_equal(frames[algo]["hits"], want["hits"]) and np.array_equal(frames[algo]["rgb"], want["rgb"]), (storage, algo)
                else:
                    close = (np.abs(frames[algo]["rgb"].astype(np.int32) - want["rgb"].astype(np.int32)) <= 1).all(-1).mean()
                    assert close >= 0.999, (storage, algo, close)
            g.close()
    s.close()


@pytest.fixture(scope="module")
def terrain512():
    return scenes.terrain(512, 1234)


@pytest.mark.timeout(900)
@pytest.mark.parametrize("storage", ["vcs", "hashtable"])
def test_config3_terrain512_4k(terrain512, golden, storage):
    """configs[2]: procedural 512^3 terrain (~32 M voxels), 3840x2160, SURVEY.md 8d-3's camera -- the bench workload itself.  Both
    structures x both algorithms against the checker (the reference's host build, else its restatement) on the same scene:
    bit-exact hit map, RGB, event counters."""
    kind = oracle_kind()
    xyz, rgb = terrain512
    po.set_lighting(kind)
    ref = build_oracle(kind, xyz, rgb, storage)
    s = _product(xyz, rgb, storage)
    assert dict(diameter=s.info()["diameter"], min_coord=s.info()["min_coord"], filled=s.info()["filled"]) == ref.info()
    for algo in ("longestaxis", "original"):
        want = _compare_frame(s, ref, config3_camera(), 3840, 2160, algo, 1, golden, f"config3_{storage}_{algo}", tag=f"config3 {storage}")
        assert 0.3 < (want["hits"][..., 3] != 0).mean() < 1.0
    s.close(); ref.close()


def orbit_camera_2048(v, w, h):
    """View v of the 64-view orbit of configs[3] (SURVEY.md 8d-4): radius 1.5 * 1024 around the centre of the 2048^3 volume, elevation 20 degrees."""
    ang = 2.0 * np.pi * (v + 0.37) / 64
    r, el = 1.5 * 1024.0, np.deg2rad(20.0)
    org = (float(1024 + r * np.cos(el) * np.cos(ang)), float(1024 + r * np.sin(el)), float(1024 + r * np.cos(el) * np.sin(ang)))
    return api.Camera(org, (1024.0, 1024.0, 1024.0), (0.0, 1.0, 0.0), 60.0, np.float32(w) / np.float32(h))


@pytest.mark.timeout(1500)
def test_config4_orbit_2048_views_match_reference_kernels(golden):
    """configs[3]: 2048^3 sparse scene (~36 M voxels, 32^3 region table), VCS, four views of the 64-view orbit at 1920x1080, both
    algorithms.  The reference crawls on this scene for seconds per frame on the GPU, so the checker is its own CUDA kernels
    compiled with -fmad=false where built, else the restatement on the host cores: bit-exact hit maps and RGB.  Also: the views
    rendered as ONE batch (the way the orbit is sharded over GPUs) equal the single renders."""
    kind = "refgx" if po.available("refgx") else "orc"
    import torch
    xyz, rgb = scenes.sparse_shells(2048, 64, seed=7, fill_pct=35)
    assert xyz.shape[0] > 30_000_000
    w, h = 1920, 1080
    views = CONFIG4_VIEWS
    cams = [orbit_camera_2048(v, w, h) for v in views]
    s = _product(xyz, rgb, "vcs")
    po.set_lighting(kind)
    ref = build_oracle(kind, xyz, rgb, "vcs")
    assert dict(diameter=s.info()["diameter"], min_coord=s.info()["min_coord"], filled=s.info()["filled"]) == ref.info()
    for algo in ("longestaxis", "original"):
        batch = torch.zeros((len(cams), h, w, 3), dtype=torch.uint8, device="cuda:0")
        s.render_views_device(w, h, algo, cams, batch.data_ptr())
        s.synchronize()
        for i, cam in enumerate(cams):
            got = s.render(w, h, algo, cam, want_hits=True)
            want = ref.render(cam.data, w, h, algo)
            nbad = int((got["hits"] != want["hits"]).any(-1).sum())
            assert nbad == 0, (algo, views[i], nbad)
            assert np.array_equal(got["rgb"], want["rgb"]), (algo, views[i])
            assert np.array_equal(batch[i].cpu().numpy(), got["rgb"]), (algo, views[i])
            assert int(want["hits"][..., 3].sum()) > 100_000
            _check_golden(golden, f"config4_view{views[i]}_vcs_{algo}", got["hits"], rgb=got["rgb"])
    s.close(); ref.close()


@pytest.mark.timeout(900)
def test_config5_incoherent_rays_1024_full_buffer(golden):
    """configs[4]: incoherent-ray stress -- one random direction per pixel of a 4K frame (8 294 400 rays, SURVEY.md 8d-5's counter-based
    hash) + shadow rays on the 1024^3 sparse scene, VCS + longest axis (and original): the FULL ray buffer against the checker's
    per-ray routines (the reference's rayMarchVoxelSceneLongestAxis / rayMarchVoxelScene in its host build, else their
    restatement): colours, hit voxels and counters."""
    kind = oracle_kind()
    xyz, rgb = scenes.sparse_shells(1024, 64, seed=11, fill_pct=35)
    rays = config5_rays()
    po.set_lighting(kind)
    s, ref = _product(xyz, rgb, "vcs"), build_oracle(kind, xyz, rgb, "vcs")
    s.set_statistics(True)
    for algo in ("longestaxis", "original"):
        got = s.trace_rays(rays, algo, want_hits=True)
        st = s.get_statistics()
        want = ref.trace_rays(rays, algo, want_counters=True, threads=CORES)
        assert np.array_equal(got["hits"], want["hits"]), (algo, int((got["hits"] != want["hits"]).any(-1).sum()))
        assert np.array_equal(got["colour"], want["colour"]), algo
        mine = [st["exist_checks"], st["exist_false"], st["lookups"], st["lookup_hits"]]
        assert mine == [int(v) for v in want["counters"][:4]], algo
        assert want["hits"][:, 3].mean() > 0.2
        _check_golden(golden, f"config5_vcs_{algo}", got["hits"], colour=got["colour"], counters=mine)
    s.close(); ref.close()


def test_one_million_single_voxel_inserts_are_cheap():
    """VERDICT r01 weak 6: a caller porting the reference's insertVoxel loop (VoxelSceneCPU.cuh:16-46).  One million single-voxel
    calls through the C ABI must cost host appends, not device allocations: the whole loop (driven from C through one ctypes call per
    voxel here) stays far below the old cost of two cudaMallocs + a stream sync per voxel, and the built scene holds every voxel."""
    import time
    n = 1_000_000
    rng = np.random.default_rng(3)
    xyz = rng.integers(-200, 200, size=(n, 3)).astype(np.int32)
    rgb = rng.integers(1, 1 << 24, size=n).astype(np.uint32)
    s = api.VoxelScene(0)
    fn, h = s.lib.vrm_scene_insert_voxel, s.h
    xs, ys, zs, cs = xyz[:, 0].tolist(), xyz[:, 1].tolist(), xyz[:, 2].tolist(), rgb.tolist()
    t0 = time.perf_counter()
    for i in range(n):
        fn(h, xs[i], ys[i], zs[i], cs[i])
    dt = time.perf_counter() - t0
    s.generate_voxel_scene("vcs")
    print(f"1 M vrm_scene_insert_voxel calls: {dt:.2f} s")
    assert dt < 5.0, dt          # ~1 us per call is the ctypes dispatch; the C side is a vector append
    # last write wins among duplicates: compare with a dictionary built in insertion order
    last = {}
    for i, key in enumerate(map(tuple, xyz[:200000].tolist())):
        last[key] = i
    full = {}
    for i, key in enumerate(zip(xs, ys, zs)):
        full[key] = cs[i]
    assert s.info()["unique_voxels"] == len(full)
    probe = np.array(list(last.keys())[:50000], np.int32)
    val, _ = s.lookup(probe)
    assert val.tolist() == [full[tuple(k)] for k in probe.tolist()]
    s.close()


def test_unaligned_hit_buffers_are_rejected_or_copied(probe):
    """ADVICE r01: hit records are 16-byte stores.  A misaligned DEVICE hit buffer is refused with a status (not a sticky fault); a
    misaligned page-locked HOST buffer silently takes the copy path and gives the same bytes."""
    import torch
    xyz, rgb = probe
    s = _product(xyz, rgb, "vcs")
    w, h = 160, 90
    cam = api.Camera.reference_default(w, h)
    want = s.render(w, h, "longestaxis", cam, scale=8, want_hits=True)
    fb = torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda:0")
    raw = torch.zeros(h * w * 4 + 4, dtype=torch.int32, device="cuda:0")
    with pytest.raises(api.VrmError):
        s.render_device(w, h, "longestaxis", cam, fb.data_ptr(), raw.data_ptr() + 4, scale=8)
    s.render_device(w, h, "longestaxis", cam, fb.data_ptr(), raw.data_ptr(), scale=8)   # the handle still works
    s.synchronize()
    assert np.array_equal(raw[: h * w * 4].cpu().numpy().reshape(h, w, 4), want["hits"])
    pinned = torch.zeros(h * w * 4 + 1, dtype=torch.int32).pin_memory()
    hits_view = pinned.numpy()[1:].reshape(h, w, 4)                                     # 4-byte aligned, not 16
    rgb_out = np.zeros((h, w, 3), np.uint8)
    import ctypes as C
    ms = C.c_float()
    rc = s.lib.vrm_render(s.h, api._ptr(cam.data), api._ptr(np.zeros(3, np.float32)), 8, api.ALGO_LONGEST_AXIS, w, h, api._ptr(rgb_out), api._ptr(hits_view), C.byref(ms))
    assert rc == 0
    assert np.array_equal(hits_view, want["hits"]) and np.array_equal(rgb_out, want["rgb"])
    s.close()


def test_large_pinned_view_batch_is_not_limited_by_the_debug_kernel(probe):
    """ADVICE r01: the 2^32 pixel-slot limit belongs to the persistent debug kernel only; the default kernels take any batch."""
    import torch
    xyz, rgb = probe
    s = _product(xyz, rgb, "vcs")
    w, h, n = 8, 4, 70000          # > 65535 views: two launches; 70 000 x 32-pixel tiles is far below any limit, the old check was on tiles * 32 * views
    cams = np.repeat(api.Camera.reference_default(w, h).data[None], n, 0)
    pinned = torch.zeros((n, h, w, 3), dtype=torch.uint8).pin_memory()
    import ctypes as C
    ms = C.c_float()
    rc = s.lib.vrm_render_views(s.h, api._ptr(np.ascontiguousarray(cams)), n, api._ptr(np.zeros(3, np.float32)), 8, api.ALGO_LONGEST_AXIS, w, h, api._ptr(pinned.numpy()), C.byref(ms))
    assert rc == 0
    one = s.render(w, h, "longestaxis", api.Camera.reference_default(w, h), scale=8)["rgb"]
    got = pinned.numpy()
    assert np.array_equal(got[0], one) and np.array_equal(got[-1], one) and np.array_equal(got[65535], one)
    s.close()
