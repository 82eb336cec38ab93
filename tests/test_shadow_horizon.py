"""CPU tier: the shadow horizon map (vrm_core.cuh HorizonView, vrm_flat.cuh FlatRay::past_horizon) on the product's traversal compiled
for the host (tests/horizon_sim.py: tests/hostsim plus the map).  Lit shadow rays that end at the map must give exactly what the full walk gives: RGB and hit maps equal to
the oracle bit for bit, with the as-executed event counters no higher than without the map."""
import numpy as np
import pytest

from tests import horizon_sim as hs
from tests.common import COMBOS, MINI_CAMERAS, PROBE_CAMERAS, build_oracle, camera, oracle_kind, po, scenes

# (1,1,1); axis-aligned; negative components; near-axis (every component >= kHorizonMinComponent); near-axis below it (no map)
LIGHTS = [(1.0, 1.0, 1.0), (0.0, 1.0, 0.0), (1.0, 0.0, 0.0), (-0.3, -0.8, 0.5), (0.3, 0.7, -0.65), (0.08, 1.0, 0.1), (0.01, 1.0, 0.02)]
FAST = 3  # sim_set_flat: the generic state machine with its warp-uniform fast paths taken per ray


@pytest.fixture
def horizon():
    hs.load()
    yield
    hs.set_form(1)
    po.set_lighting(oracle_kind())


def _light(kind, direction):
    d = po.unit_vector(direction, kind)
    po.set_lighting(kind, direction=d)
    hs.set_lighting(d)


def _terrain_slice(seed=1234):
    """A 128^2 piece of the bench terrain, 48 voxels high, under a region table four regions tall (one marker voxel high above it):
    like the bench scene, lit shadow rays leave the terrain into empty clusters and null regions."""
    xyz, rgb = scenes.terrain(128, seed, max_height=48)
    return np.concatenate([xyz, np.array([[127, 250, 127]], xyz.dtype)]), np.concatenate([rgb, rgb[:1]])


SLICE_CAMERAS = [((230.0, 140.0, 210.0), (64.0, 20.0, 64.0), 60.0), ((-60.0, 120.0, 190.0), (64.0, 20.0, 64.0), 50.0)]


def _check_scene(xyz, rgb, cams, w, h, scale, combos):
    kind = oracle_kind()
    for storage, algo in combos:
        a, b = build_oracle(kind, xyz, rgb, storage), hs.Scene(xyz, rgb, storage)
        for o, l, fov in cams:
            cam = camera(o, l, fov, w, h, kind)
            ref = a.render(cam, w, h, algo, scale=scale)
            off = b.render(cam, w, h, algo, scale=scale, horizon=False)
            on = b.render(cam, w, h, algo, scale=scale, horizon=True)
            for k in ("rgb", "hits"):
                assert np.array_equal(on[k], ref[k]), (storage, algo, k, o)
            assert np.all(on["counters"] <= off["counters"]), (storage, algo, on["counters"], off["counters"])


@pytest.mark.parametrize("light", LIGHTS)
def test_horizon_probe_and_mini_match_oracle(horizon, light):
    hs.set_form(FAST)
    _light(oracle_kind(), light)
    _check_scene(*scenes.probe_scene(), PROBE_CAMERAS, 160, 90, 8, COMBOS)
    _check_scene(*scenes.mini_scene(), MINI_CAMERAS, 128, 72, 1, COMBOS)


@pytest.mark.parametrize("form", [FAST, 1])
@pytest.mark.parametrize("light", [(1.0, 1.0, 1.0), (-0.3, -0.8, 0.5), (0.0, 1.0, 0.0)])
def test_horizon_terrain_slice_matches_oracle(horizon, form, light):
    hs.set_form(form)
    _light(oracle_kind(), light)
    _check_scene(*_terrain_slice(), SLICE_CAMERAS, 192, 108, 1, [("vcs", "longestaxis"), ("vcs", "original")])


def test_horizon_saves_work_on_terrain(horizon):
    """The map must actually end shadow rays early on the kind of scene it is for (as-executed exist checks go down; most of what it
    saves are null-region skips, which no counter sees)."""
    hs.set_form(FAST)
    _light(oracle_kind(), (1.0, 1.0, 1.0))
    b = hs.Scene(*_terrain_slice())
    cam = camera(*SLICE_CAMERAS[0], 192, 108)
    off = b.render(cam, 192, 108, "longestaxis", horizon=False)
    on = b.render(cam, 192, 108, "longestaxis", horizon=True)
    assert on["counters"][0] < off["counters"][0], (on["counters"], off["counters"])


def _surface_rays(xyz, n, rng):
    """Rays from random points above the scene towards random stored voxels: their hits are spread over the surface."""
    tgt = xyz[rng.integers(0, len(xyz), n)].astype(np.float64) + 0.5
    org = tgt + rng.normal(size=(n, 3)) * 40.0
    org[:, 1] = np.abs(org[:, 1]) + 60.0
    d = tgt - org
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.concatenate([org, d], axis=1).astype(np.float32)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("algo", ["longestaxis", "original"])
def test_horizon_threshold_is_beyond_every_occupied_test(horizon, seed, algo):
    """Random surface shadow rays and lights, every shadow ray marched in full: no voxel test that finds an occupied cluster happens
    once the ray is past the threshold its one map lookup gave it."""
    rng = np.random.default_rng(seed)
    xyz, rgb = _terrain_slice(1000 + seed)
    b = hs.Scene(xyz, rgb)
    checked = passed = 0
    for _ in range(6):
        while True:
            v = rng.normal(size=3)
            v[1] = abs(v[1]) + 0.2
            u = v / np.linalg.norm(v)
            if np.all(np.abs(u) >= 0.0625):
                break
        _light("orc", tuple(v))
        res = b.property(_surface_rays(xyz, 4000, rng), algo)
        assert res is not None
        rays_n, bad, past, found = res
        assert bad == 0, (v, rays_n, bad, past, found)
        checked += rays_n; passed += past
    assert checked > 5000 and passed > checked // 10, (checked, passed)
