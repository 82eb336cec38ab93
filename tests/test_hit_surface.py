"""CPU tier: the hit-surface definition (vrm_core.cuh primary_ray + hit_surface, the function the vrm_hit_surface_* kernel runs) built for
the host, against its numpy fp32 restatement in tests/surface_ref.py, bit for bit, on the oracle's hit maps and traced rays."""
import numpy as np
import pytest

from tests import surface_ref as sr
from tests.common import COMBOS, PROBE_CAMERAS, build_oracle, camera, oracle_kind, po
from voxelraymarcher_b200 import scenes

W, H = 160, 90
SCALE = 8
TRANSLATIONS = [(0.0, 0.0, 0.0), (0.75, -1.25, 2.5)]
# Worst distance (local voxel units) of the exact entry point s + t D from the reported voxel's box over the inputs below, per algorithm.
# It measures how far from the exact ray the reference walk reports its voxel; it is not a tolerance on depth or face, which must match
# bit for bit.  Measured on these inputs: original 2.7e-5 (accumulated fp32 rounding; 0.26 once, VCS with the translation), longest
# axis 0.9999 -- that walk steps along the longest axis and can report a face neighbour of the voxel the exact ray enters.
DRIFT_BOUND = {"original": 0.5, "longestaxis": 1.5}


@pytest.fixture(scope="module")
def oracles():
    kind = oracle_kind()
    po.set_lighting(kind)
    xyz, rgb = scenes.probe_scene()
    out = {st: build_oracle(kind, xyz, rgb, st) for st in ("hashtable", "vcs")}
    yield kind, out
    for s in out.values():
        s.close()


def _trace_rays(seed=5):
    """Rays towards the probe scene (world units at scale 8) with negative, zero and axis-aligned direction components."""
    rng = np.random.default_rng(seed)
    n = 4000
    org = rng.uniform(-6.0, 18.0, (n, 3)).astype(np.float32)
    target = rng.uniform(-2.0, 14.0, (n, 3)).astype(np.float32)
    d = (target - org).astype(np.float32)
    d[n // 4: n // 2, rng.integers(0, 3)] = 0.0                      # one zero component
    d[n // 2: 5 * n // 8, :] = 0.0
    axis = rng.integers(0, 3, n // 8)
    d[np.arange(n // 2, 5 * n // 8), axis] = np.where(rng.random(n // 8) < 0.5, -1.0, 1.0)  # axis-aligned
    d[5 * n // 8:, 1] = -np.abs(d[5 * n // 8:, 1])                    # downwards, onto the floor
    length = np.sqrt((d.astype(np.float64) ** 2).sum(1)).astype(np.float32)
    d = (d / np.maximum(length, np.float32(1e-6))[:, None]).astype(np.float32)
    d[~np.isfinite(d).all(1)] = (0.0, -1.0, 0.0)
    return np.concatenate([org, d], 1).astype(np.float32)


def test_numpy_pixel_rays_equal_primary_ray():
    for o, l, fov in PROBE_CAMERAS:
        cam = camera(o, l, fov, W, H, "orc")
        rays = np.zeros((H * W, 6), np.float32)
        length = np.zeros(H * W, np.float32)
        sr.load().surf_pixel_rays(sr._p(cam), W, H, sr._p(rays), sr._p(length))
        P, D, ln = sr.pixel_rays(cam, W, H)
        assert sr.same_bits(P.reshape(-1, 3), rays[:, :3]) and sr.same_bits(D.reshape(-1, 3), rays[:, 3:])
        assert sr.same_bits(ln.reshape(-1), length)


@pytest.mark.parametrize("storage,algorithm", COMBOS)
@pytest.mark.parametrize("translation", TRANSLATIONS)
def test_views_on_oracle_hit_maps(oracles, storage, algorithm, translation):
    kind, ref = oracles
    cams = [camera(o, l, fov, W, H, kind) for o, l, fov in PROBE_CAMERAS]   # the last one starts far outside: scene-entry loop
    hits = np.stack([ref[storage].render(c, W, H, algorithm, scale=SCALE, translation=translation)["hits"] for c in cams])
    assert hits[..., 3].sum() > 1000
    want_d, want_f = sr.views(hits, cams, W, H, SCALE, translation)
    got_d, got_f = sr.sim_views(hits, cams, W, H, SCALE, translation)
    assert sr.same_bits(got_d, want_d)
    assert np.array_equal(got_f, want_f)
    flag = hits[..., 3] != 0
    assert np.isinf(got_d[~flag]).all() and (got_f[~flag] == 0).all()
    assert np.isfinite(got_d[flag]).all() and ((got_f[flag] >= 1) & (got_f[flag] <= 6)).all()
    worst = 0.0
    for v, c in enumerate(cams):
        P, D, _ = sr.pixel_rays(c, W, H)
        worst = max(worst, float(sr.entry_distance(hits[v], P, D, translation, SCALE).max(initial=0.0)))
    assert worst < DRIFT_BOUND[algorithm], worst


@pytest.mark.parametrize("storage,algorithm", COMBOS)
@pytest.mark.parametrize("translation", TRANSLATIONS)
def test_rays_on_oracle_traces(oracles, storage, algorithm, translation):
    _, ref = oracles
    rays = _trace_rays()
    hits = ref[storage].trace_rays(rays, algorithm, scale=SCALE, translation=translation)["hits"]
    assert hits[:, 3].sum() > 500
    want_d, want_f = sr.rays(hits, rays, SCALE, translation)
    got_d, got_f = sr.sim_rays(hits, rays, SCALE, translation)
    assert sr.same_bits(got_d, want_d)
    assert np.array_equal(got_f, want_f)
    worst = float(sr.entry_distance(hits, rays[:, :3], rays[:, 3:], translation, SCALE).max(initial=0.0))
    assert worst < DRIFT_BOUND[algorithm], worst


def test_definition_edges():
    """Misses, ties (strict >: the earlier axis wins), a zero direction, origins inside the voxel and signed zeros."""
    hits = np.array([[0, 0, 0, 0],          # miss
                     [1, 1, 1, 1],          # diagonal ray from the origin: t_x == t_y == t_z -> x face
                     [0, 0, 0, 1],          # origin inside the voxel: negative depth
                     [5, 0, 0, 1],          # zero direction: NaN, face 0
                     [-1, 2, 3, 1],         # negative direction on x: face +x
                     [0, 0, 0, 1]], np.int32)
    rays = np.array([[0, 0, 0, 1, 0, 0],
                     [0, 0, 0, 0.57735026, 0.57735026, 0.57735026],
                     [0.5, 0.5, 0.5, 0, 1, 0],
                     [0, 0, 0, 0, 0, 0],
                     [3, 2.5, 3.5, -1, 0, 0],
                     [0, 0, 0, 0, 0, -1]], np.float32)
    want_d, want_f = sr.rays(hits, rays)
    got_d, got_f = sr.sim_rays(hits, rays)
    assert sr.same_bits(got_d, want_d) and np.array_equal(got_f, want_f)
    assert np.isinf(got_d[0]) and got_f[0] == 0
    assert got_f[1] == 1
    assert got_d[2] == -0.5 and got_f[2] == 3
    assert np.isnan(got_d[3]) and got_f[3] == 0
    assert got_d[4] == 3.0 and got_f[4] == 2
    assert got_f[5] == 6 and got_d[5].tobytes() == np.float32(-1.0).tobytes()
