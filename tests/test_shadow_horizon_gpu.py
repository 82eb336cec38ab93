"""GPU tier (pytest -m gpu): the shadow horizon map on the real kernels.  A handle created with VRM_SHADOW_HORIZON=0 walks every lit
shadow ray out of the scene; the default handle ends it at the map.  Frames, hit maps, trace_rays colours and reference-comparable
counters must be bit-identical between the two."""
import os

import numpy as np
import pytest

import bench
from voxelraymarcher_b200 import api, scenes

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _handle(horizon, fill, storage="vcs", light=None):
    old = os.environ.get("VRM_SHADOW_HORIZON")
    os.environ["VRM_SHADOW_HORIZON"] = "1" if horizon else "0"
    try:
        s = api.VoxelScene(0)
    finally:
        if old is None:
            del os.environ["VRM_SHADOW_HORIZON"]
        else:
            os.environ["VRM_SHADOW_HORIZON"] = old
    s.set_stream(torch.cuda.current_stream().cuda_stream)
    fill(s)
    if light is not None:
        s.setup_constant_values(**light)
    s.generate_voxel_scene(storage)
    return s


def _frame(s, w, h, cam, hits=False):
    rgb = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
    hit = torch.empty((h, w, 4), dtype=torch.int32, device="cuda") if hits else None
    s.render_device(w, h, "longestaxis", cam, rgb.data_ptr(), hit.data_ptr() if hits else None)
    torch.cuda.synchronize()
    return rgb, hit


def _same_frames(a, b, w, h, cams, hits_every=8):
    for i, cam in enumerate(cams):
        fa, ha = _frame(a, w, h, cam, hits=i % hits_every == 0)
        fb, hb = _frame(b, w, h, cam, hits=i % hits_every == 0)
        assert torch.equal(fa, fb), f"view {i}: frames differ"
        if ha is not None:
            assert torch.equal(ha, hb), f"view {i}: hit maps differ"


def _terrain(s):
    s.generate_terrain(bench.SCENE_SIZE, bench.SCENE_SEED)


@pytest.fixture(scope="module")
def terrain_pair():
    return _handle(True, _terrain), _handle(False, _terrain)


def test_terrain_4k_all_orbit_views(terrain_pair):
    on, off = terrain_pair
    _same_frames(on, off, bench.WIDTH, bench.HEIGHT, [bench.orbit_camera(api, v) for v in range(bench.ORBIT_VIEWS)])


def test_shells_2048_orbit_views():
    fill = lambda s: s.generate_sparse_shells(2048, 64, 7, 35)  # noqa: E731
    on, off = _handle(True, fill), _handle(False, fill)
    cams = bench.orbit_views_2048(api, 1920, 1080)
    _same_frames(on, off, 1920, 1080, [cams[v] for v in (0, 16, 32, 48)], hits_every=1)


def test_config5_trace_rays():
    fill = lambda s: s.generate_sparse_shells(1024, 64, 11, 35)  # noqa: E731
    on, off = _handle(True, fill), _handle(False, fill)
    rays = scenes.random_rays(1 << 21, (512.0 + 31.5, 512.0 + 31.5, 512.0 + 31.5), seed=42)
    a, b = on.trace_rays(rays, "longestaxis", want_hits=True), off.trace_rays(rays, "longestaxis", want_hits=True)
    for k in ("colour", "hits"):
        assert np.array_equal(a[k], b[k]), k


LIGHTS = [dict(light_direction=api.make_unit_vector((0.2, 0.9, -0.38)), light_color=(1.0, 0.8, 0.6)),
          dict(light_direction=api.make_unit_vector((-0.3, 0.8, -0.5))),
          dict(light_direction=(0.0, 1.0, 0.0)),
          dict(light_direction=api.make_unit_vector((0.08, 1.0, 0.1))),
          dict(use_point_light=True, light_position=(60.0, 90.0, 80.0)),
          dict(use_shadows=False)]


@pytest.mark.parametrize("light", LIGHTS)
def test_lighting_variants(light):
    on, off = _handle(True, _terrain, light=light), _handle(False, _terrain, light=light)
    _same_frames(on, off, 1920, 1080, [bench.orbit_camera(api, v) for v in (0, 13, 40)], hits_every=1)


@pytest.mark.parametrize("light", LIGHTS[:3])
def test_set_lighting_on_built_scene(terrain_pair, light):
    """The map follows the light: set_lighting on a built scene rebuilds it (and dropping shadows drops it)."""
    on, off = terrain_pair
    try:
        for s in (on, off):
            s.setup_constant_values(use_shadows=False)
            s.setup_constant_values(**light)
        fresh = _handle(True, _terrain, light=light)
        cams = [bench.orbit_camera(api, v) for v in (0, 29)]
        _same_frames(on, off, 1920, 1080, cams, hits_every=1)
        _same_frames(on, fresh, 1920, 1080, cams, hits_every=1)
    finally:
        for s in (on, off):
            s.setup_constant_values()


def test_reference_counters_unchanged_and_executed_work_lower(terrain_pair):
    on, off = terrain_pair
    cam = bench.orbit_camera(api, 0)
    got = {}
    for mode in ("reference", "executed"):
        for name, s in (("on", on), ("off", off)):
            s.set_statistics(True, as_executed=mode == "executed")
            _frame(s, 1920, 1080, cam)
            got[(mode, name)] = s.get_statistics()
            s.set_statistics(False)
    assert got[("reference", "on")] == got[("reference", "off")]
    ex_on, ex_off = got[("executed", "on")], got[("executed", "off")]
    assert all(ex_on[k] <= ex_off[k] for k in ex_off), (ex_on, ex_off)
