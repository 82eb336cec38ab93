"""CPU tier: the exact ray cast (vrm_core.cuh cast_ray, the function the vrm_cast_* kernel runs, with its exact leaps) built for the host,
against the numpy cell-by-cell walk of tests/cast_ref.py, bit for bit, on both storage types."""
import numpy as np
import pytest

from tests import cast_ref as cr
from tests import surface_ref as sr
from tests.common import MINI_CAMERAS, PROBE_CAMERAS, camera
from voxelraymarcher_b200 import scenes

W, H = 96, 54
# (scene, scale, translation): the probe scene is cast at scale 8, the others in voxel units
SCENES = {
    "probe": (scenes.probe_scene, 8, (0.0, 0.0, 0.0)),
    "probe_translated": (scenes.probe_scene, 8, (0.75, -1.25, 2.5)),
    "mini": (scenes.mini_scene, 1, (0.0, 0.0, 0.0)),
    "terrain192": (lambda: scenes.terrain(192), 1, (0.0, 0.0, 0.0)),
    "shells512": (lambda: scenes.sparse_shells(512), 1, (0.0, 0.0, 0.0)),
}
_CACHE = {}


def scene(name):
    """(Stored, {storage: Sim}, scale, translation), built once per module run."""
    if name not in _CACHE:
        fn, scale, tr = SCENES[name]
        if name == "probe_translated" and "probe" in _CACHE:
            st, sims = _CACHE["probe"][:2]
        else:
            xyz, rgb = fn()
            st, sims = cr.Stored(xyz, rgb), {s: cr.Sim(xyz, rgb, s) for s in ("vcs", "hashtable")}
        _CACHE[name] = (st, sims, scale, tr)
    return _CACHE[name]


def check_properties(got, rays, ranges, sim, scale, translation):
    hit = got["hits"][:, 3] != 0
    entered = hit & (got["face"] != 0)
    # depth of an entered-cell hit == hit_surface of the same record; the face too, except in exact ties between axes
    want_d, want_f = sr.rays(got["hits"], rays, scale, translation)
    assert np.array_equal(got["depth"][entered], want_d[entered])
    hits = got["hits"][entered]
    P = rays[entered, :3]
    D = rays[entered, 3:]
    s = (np.float32(scale) * (P - np.asarray(translation, np.float32))).astype(np.float32)
    with np.errstate(all="ignore"):
        ta = [np.where(D[:, a] != 0, ((np.where(D[:, a] > 0, hits[:, a], hits[:, a] + 1).astype(np.float32) - s[:, a]) / D[:, a]).astype(np.float32),
                       -np.inf) for a in range(3)]
    tmax = np.maximum(np.maximum(ta[0], ta[1]), ta[2])
    tie = sum((t == tmax).astype(int) for t in ta) > 1
    assert np.array_equal(got["face"][entered][~tie], want_f[entered][~tie])
    assert sr.same_bits(got["depth"][entered][~tie], want_d[entered][~tie])   # a tie at tau = 0 may differ in the sign of zero
    # the colour is what a lookup of the hit returns; misses are +inf / 0 / EMPTY
    assert np.array_equal(got["colour"][hit], sim.lookup(got["hits"][hit, :3]))
    assert np.isposinf(got["depth"][~hit]).all() and (got["face"][~hit] == 0).all() and (got["colour"][~hit] == cr.EMPTY).all()
    if ranges is not None:
        start = hit & (got["face"] == 0)
        assert sr.same_bits(got["depth"][start], ranges[start, 0])
    return int(hit.sum()), int(tie.sum())


@pytest.mark.parametrize("name", list(SCENES))
def test_rays_match_numpy_walk(name):
    st, sims, scale, tr = scene(name)
    cases = cr.ray_cases(st, scale, tr, seed=len(name), n=800 if name in ("terrain192", "shells512") else 1500)
    total_hits = 0
    for case, rays in cases.items():
        for rname, ranges in cr.range_cases(len(rays)).items():
            if case not in ("random", "ties") and rname not in ("default", "interval"):
                continue
            want = cr.cast_rays(st, rays, ranges, scale, tr)
            vcs = sims["vcs"].cast_rays(rays, ranges, scale, tr)
            hsh = sims["hashtable"].cast_rays(rays, ranges, scale, tr)
            for got, storage in ((vcs, "vcs"), (hsh, "hashtable")):
                assert cr.same(got, want), (name, case, rname, storage)
            assert cr.same(vcs, hsh)
            nh, _ = check_properties(vcs, rays, ranges, sims["vcs"], scale, tr)
            total_hits += nh
            if rname == "default" and case in ("random", "ties", "planes", "inside", "far"):
                assert nh > 0, (name, case)
    assert total_hits > 1000


@pytest.mark.parametrize("name", ["probe", "probe_translated", "mini"])
def test_views_match_numpy_walk(name):
    st, sims, scale, tr = scene(name)
    cams = [camera(o, l, fov, W, H, "orc") for o, l, fov in (PROBE_CAMERAS if name.startswith("probe") else MINI_CAMERAS)]
    want = cr.cast_views(st, cams, W, H, scale, tr)
    assert want["hits"][..., 3].sum() > 500
    for storage in ("vcs", "hashtable"):
        got = sims[storage].cast_views(cams, W, H, scale, tr)
        assert cr.same(got, want), storage
    # depth of an entered-cell hit == len + the hit surface's depth
    want_d, _ = sr.views(want["hits"], cams, W, H, scale, tr)
    entered = (want["hits"][..., 3] != 0) & (want["face"] != 0)
    assert sr.same_bits(want["depth"][entered], want_d[entered])


def test_skip_to_box_matches_plain_stepping():
    """The numpy walk's skip to the box entry (per-axis rule) against stepping through the cells outside the box, origins 1..300 cells out."""
    for name in ("mini", "probe_translated"):
        st, sims, scale, tr = scene(name)
        rays = cr.moderate_rays(st, scale, tr)
        skip = cr.cast_rays(st, rays, None, scale, tr)
        step = cr.cast_rays(st, rays, None, scale, tr, skip_far=False, margin=600)
        assert cr.same(skip, step)
        assert skip["hits"][:, 3].sum() > 100
        assert cr.same(sims["vcs"].cast_rays(rays, None, scale, tr), skip)


def test_t_far_at_depth_is_inclusive():
    """Scale 1: an interval ending at the hit's depth still finds it, one ulp shorter does not return it."""
    st, sims, scale, tr = scene("mini")
    rays = cr.ray_cases(st, 1, tr, seed=9)["random"]
    sim = sims["vcs"]
    full = sim.cast_rays(rays)
    entered = (full["hits"][:, 3] != 0) & (full["face"] != 0)
    assert entered.sum() > 300
    r, d = rays[entered], full["depth"][entered]
    at = sim.cast_rays(r, np.stack([np.zeros_like(d), d], 1))
    assert np.array_equal(at["hits"], full["hits"][entered]) and sr.same_bits(at["depth"], d)
    short = sim.cast_rays(r, np.stack([np.zeros_like(d), np.nextafter(d, np.float32(-np.inf))], 1))
    assert not (np.all(short["hits"] == full["hits"][entered], 1) & (short["hits"][:, 3] != 0)).any()
    assert cr.same(short, cr.cast_rays(st, r, np.stack([np.zeros_like(d), np.nextafter(d, np.float32(-np.inf))], 1)))


def test_definition_edges():
    """Zero direction (start cell only), start-cell hits at t_near, and the rays that are always misses."""
    xyz = np.array([[2, 3, 4], [10, 3, 4]], np.int32)
    rgb = np.array([cr.EMPTY, 0x123456], np.uint32)        # a voxel stored with the colour EMPTY is hit
    st = cr.Stored(xyz, rgb)
    sim = cr.Sim(xyz, rgb, "vcs")
    nan, inf = np.nan, np.inf
    rays = np.array([[2.5, 3.5, 4.5, 0, 0, 0],          # zero direction inside a voxel: start-cell hit
                     [5.5, 3.5, 4.5, 0, 0, 0],          # zero direction in empty space: miss
                     [0.5, 3.5, 4.5, 1, 0, 0],          # hits (2, 3, 4) through -x at t = 1.5
                     [12.5, 3.5, 4.5, -2, 0, 0],        # hits (10, 3, 4) through +x at t = 0.75
                     [0.5, 3.5, 4.5, -0.0, 0, 0],       # -0.0 is zero: miss
                     [nan, 3.5, 4.5, 1, 0, 0],          # non-finite origin
                     [0.5, 3.5, 4.5, inf, 0, 0]],       # non-finite direction
                    np.float32)
    ranges = np.array([[0.25, 1], [0, inf], [0, inf], [0, inf], [0, inf], [0, inf], [0, inf]], np.float32)
    got = sim.cast_rays(rays, ranges)
    assert cr.same(got, cr.cast_rays(st, rays, ranges))
    assert got["hits"][0].tolist() == [2, 3, 4, 1] and got["face"][0] == 0 and got["depth"][0] == np.float32(0.25)
    assert got["colour"][0] == cr.EMPTY
    assert got["hits"][2].tolist() == [2, 3, 4, 1] and got["face"][2] == 1 and got["depth"][2] == np.float32(1.5)
    assert got["hits"][3].tolist() == [10, 3, 4, 1] and got["face"][3] == 2 and got["depth"][3] == np.float32(0.75)
    assert got["colour"][3] == 0x123456
    for i in (1, 4, 5, 6):
        assert got["hits"][i, 3] == 0 and np.isposinf(got["depth"][i]) and got["colour"][i] == cr.EMPTY
