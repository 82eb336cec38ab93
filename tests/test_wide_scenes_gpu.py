"""GPU tier (pytest -m gpu): the wide region tables of tests/test_wide_scenes.py on the real kernels.  Renders and traces of every storage x
algorithm combination against the oracle at scales 1, 3, 8 and 100 (D = 26, 200, 512, and both D = 1024 tables with a bounded ray count),
the shadow horizon map on and off where its cells are 16 and 32 voxels wide, exact casts and hit surfaces against tests/cast_ref.py and
tests/surface_ref.py, and every selectable render and trace form once on a wide table."""
import os

import numpy as np
import pytest

from tests import cast_ref as cr
from tests import surface_ref as sr
from tests.common import COMBOS, build_oracle, horizon_grid, po
from tests.test_kernel_forms_gpu import RENDER_FORMS, SWITCHES, TRACE_FORMS
from tests.test_wide_scenes import KIND, WIDE_CASTS, cast_cases, scene, wide_cameras, wide_rays
from voxelraymarcher_b200 import api

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

GW, GH = 160, 90
# scale -> translation (world units; the scenes' cameras and rays are placed to match)
SCALES = {1: (0.0, 0.0, 0.0), 3: (-40000.5, 1234.25, 60000.0), 8: (0.75, -1.25, 2.5), 100: (-7.25, 50.5, 8.0)}
COUNTER_KEYS = ("exist_checks", "exist_false", "lookups", "lookup_hits")


def cam(o, l, fov, w, h):
    return api.Camera(o, l, (0.0, 1.0, 0.0), fov, np.float32(w) / np.float32(h))


def gpu_scene(name, storage, env=None, light=None):
    """A scene built with exactly the switches in env (read at vrm_scene_create) and the given light (unit (1, 1, 1) when None)."""
    saved = {k: os.environ.pop(k) for k in SWITCHES + ("VRM_SHADOW_HORIZON",) if k in os.environ}
    os.environ.update(env or {})
    try:
        s = api.VoxelScene(0)
    finally:
        for k in env or {}:
            del os.environ[k]
        os.environ.update(saved)
    xyz, rgb, _ = scene(name)
    s.add_voxels(xyz, rgb)
    if light is not None:
        s.setup_constant_values(light_direction=light)
    s.generate_voxel_scene(storage)
    return s


class Oracle:
    """Oracle scenes built once per (scene, storage); the light is set per call."""

    def __init__(self):
        self.built = {}

    def get(self, name, storage):
        if (name, storage) not in self.built:
            for k in [k for k in self.built if k[0] != name]:         # one wide table at a time (D = 1024: an 8 GiB virtual calloc)
                self.built.pop(k).close()
            xyz, rgb, _ = scene(name)
            self.built[(name, storage)] = build_oracle(KIND, xyz, rgb, storage)
        return self.built[(name, storage)]

    def close(self):
        for r in self.built.values():
            r.close()


@pytest.fixture(scope="module")
def oracle():
    o = Oracle()
    yield o
    o.close()
    po.set_lighting(KIND)


def check_against_oracle(s, ref, name, algo, scale, tr, n_rays, w=GW, h=GH, counters=True):
    tag = (name, algo, scale)
    hit_px = 0
    for o, l, fov in wide_cameras(name, scale, tr):
        c = cam(o, l, fov, w, h)
        want = ref.render(c.data, w, h, algo, scale=scale, translation=tr)
        got = s.render(w, h, algo, c, scale=scale, translation=tr, want_hits=True)
        assert np.array_equal(got["hits"], want["hits"]), tag + (o, int((got["hits"] != want["hits"]).any(-1).sum()))
        assert np.array_equal(got["rgb"], want["rgb"]), tag + (o,)
        hit_px += int((want["hits"][..., 3] != 0).sum())
    assert hit_px > w * h // 8, tag                  # the cameras see the pieces
    rays = wide_rays(name, n_rays, seed=scale + 17, scale=scale, translation=tr)
    want = ref.trace_rays(rays, algo, scale=scale, translation=tr, want_counters=counters)
    s.set_statistics(counters)
    got = s.trace_rays(rays, algo, scale=scale, translation=tr, want_hits=True)
    st = s.get_statistics() if counters else None
    s.set_statistics(False)
    assert np.array_equal(got["hits"], want["hits"]), tag + (int((got["hits"] != want["hits"]).any(-1).sum()),)
    assert np.array_equal(got["colour"], want["colour"]), tag
    if counters:
        assert [st[k] for k in COUNTER_KEYS] == [int(v) for v in want["counters"][:4]], tag
    assert (want["hits"][:, 3] != 0).sum() > n_rays // 2
    return rays, got


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("scale", sorted(SCALES))
@pytest.mark.parametrize("storage,algo", COMBOS)
@pytest.mark.parametrize("name", ["d26", "d200", "d512"])
def test_wide_renders_and_traces_match_oracle(oracle, name, storage, algo, scale):
    """Hit maps, RGB, trace colours, hit records and reference-comparable counters bit for bit with the oracle: cameras inside the table, at
    its far corner and 10^3 .. 10^5 voxels out; rays from far outside, face to face and from table-relative coordinates above 2^15."""
    tr = SCALES[scale]
    po.set_lighting(KIND)
    s = gpu_scene(name, storage)
    check_against_oracle(s, oracle.get(name, storage), name, algo, scale, tr, 1500)
    s.close()


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("storage", ["vcs", "hashtable"])
@pytest.mark.parametrize("name", ["d1024lo", "d1024hi"])
def test_d1024_tables_match_oracle(oracle, name, storage):
    """D = 1024 with content at x = -65472 (min_coord -1023) or at x = 65535 (0 .. 1023): small renders and a bounded ray set, rays from
    outside the table that cross it included, of both algorithms, against the oracle (its table is an 8 GiB virtual calloc)."""
    po.set_lighting(KIND)
    s = gpu_scene(name, storage)
    for algo in ("longestaxis", "original"):
        check_against_oracle(s, oracle.get(name, storage), name, algo, 1, (0.0, 0.0, 0.0), 400, w=64, h=36)
    s.close()


def horizon_pair(name, storage, light):
    return gpu_scene(name, storage, {"VRM_SHADOW_HORIZON": "1"}, light), gpu_scene(name, storage, {"VRM_SHADOW_HORIZON": "0"}, light)


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("storage", ["vcs", "hashtable"])
@pytest.mark.parametrize("name", ["d200", "d512"])
def test_horizon_map_on_and_off(oracle, name, storage):
    """Handles with the map (cells of 16 and 32 voxels) and without: frames and hit maps at 640x360, trace colours and hit records, and the
    reference-comparable counters identical; as-executed counters no higher with the map; the map's render equals the oracle at 160x90."""
    D = {"d200": 200, "d512": 512}[name]
    w, h = 640, 360
    for light in ((1.0, 1.0, 1.0), (-0.3, -0.8, 0.5), (0.0, 1.0, 0.0)):
        d = po.unit_vector(light, KIND)
        assert horizon_grid(d, D)[0] > 8 or light == (0.0, 1.0, 0.0)
        on, off = horizon_pair(name, storage, d)
        po.set_lighting(KIND, direction=d)
        ref = oracle.get(name, storage)
        rays = wide_rays(name, 4000, seed=D)
        for algo in ("longestaxis", "original"):
            tag = (name, storage, light, algo)
            for o, l, fov in wide_cameras(name):
                c = cam(o, l, fov, w, h)
                a = on.render(w, h, algo, c, want_hits=True)
                b = off.render(w, h, algo, c, want_hits=True)
                assert np.array_equal(a["rgb"], b["rgb"]) and np.array_equal(a["hits"], b["hits"]), tag + (o,)
                small = cam(o, l, fov, GW, GH)
                want = ref.render(small.data, GW, GH, algo)
                got = on.render(GW, GH, algo, small, want_hits=True)
                assert np.array_equal(got["rgb"], want["rgb"]) and np.array_equal(got["hits"], want["hits"]), tag + (o, "oracle")
            ta, tb = on.trace_rays(rays, algo, want_hits=True), off.trace_rays(rays, algo, want_hits=True)
            assert np.array_equal(ta["colour"], tb["colour"]) and np.array_equal(ta["hits"], tb["hits"]), tag
            c = cam(*wide_cameras(name)[0], w, h)
            got = {}
            for mode in ("reference", "executed"):
                for key, s in (("on", on), ("off", off)):
                    s.set_statistics(True, as_executed=mode == "executed")
                    s.render(w, h, algo, c)
                    got[(mode, key)] = s.get_statistics()
                    s.set_statistics(False)
            assert got[("reference", "on")] == got[("reference", "off")], tag
            assert all(got[("executed", "on")][k] <= got[("executed", "off")][k] for k in COUNTER_KEYS), tag
        on.close()
        off.close()


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("storage", ["vcs", "hashtable"])
@pytest.mark.parametrize("name,scale,translation", WIDE_CASTS, ids=[f"{n}-scale{s}" for n, s, _ in WIDE_CASTS])
def test_wide_casts_and_hit_surfaces(name, scale, translation, storage):
    """cast_rays against the cell-by-cell walk (intervals starting and ending in long null runs, rays entering from far outside), cast_views
    on the D = 26 table, and hit_surface_rays / hit_surface_views of traced rays and rendered hit maps against surface_ref, bit for bit."""
    xyz, rgb, _ = scene(name)
    st = cr.Stored(xyz, rgb)
    s = gpu_scene(name, storage)
    for case, (rays, ranges) in cast_cases(name, 500, seed=scale + len(name), scale=scale, translation=translation).items():
        got = s.cast_rays(rays, ranges, scale, translation)
        assert cr.same(got, cr.cast_rays(st, rays, ranges, scale, translation)), (name, scale, case, storage)
    cams = wide_cameras(name, scale, translation)
    w, h = 48, 27
    if name == "d26":
        cs = [cam(o, l, fov, w, h) for o, l, fov in cams]
        assert cr.same(s.cast_views(cs, w, h, scale, translation), cr.cast_views(st, [c.data for c in cs], w, h, scale, translation))
    rays = wide_rays(name, 1000, seed=scale, scale=scale, translation=translation)
    traced = s.trace_rays(rays, "longestaxis", scale=scale, translation=translation, want_hits=True)
    assert (traced["hits"][:, 3] != 0).sum() > 600
    depth, face = s.hit_surface_rays(traced["hits"], rays, scale, translation)
    want_d, want_f = sr.rays(traced["hits"], rays, scale, translation)
    assert sr.same_bits(depth, want_d) and np.array_equal(face, want_f), (name, scale, storage)
    cs = [cam(o, l, fov, GW, GH) for o, l, fov in cams]
    hits = np.stack([s.render(GW, GH, "original", c, scale=scale, translation=translation, want_hits=True)["hits"] for c in cs])
    depth, face = s.hit_surface_views(hits, cs, GW, GH, scale, translation)
    want_d, want_f = sr.views(hits, [c.data for c in cs], GW, GH, scale, translation)
    assert sr.same_bits(depth, want_d) and np.array_equal(face, want_f), (name, scale, storage)
    s.close()


FORM_SCALE = 3


@pytest.fixture(scope="module")
def default_outputs():
    """The default forms' frames and traces on D = 200 at scale 3, per combination (computed once)."""
    out = {}
    tr = SCALES[FORM_SCALE]
    rays = wide_rays("d200", 3000, seed=5, scale=FORM_SCALE, translation=tr)
    for storage, algo in COMBOS:
        s = gpu_scene("d200", storage)
        frames = [s.render(GW, GH, algo, cam(o, l, fov, GW, GH), scale=FORM_SCALE, translation=tr, want_hits=True)
                  for o, l, fov in wide_cameras("d200", FORM_SCALE, tr)]
        out[(storage, algo)] = (frames, s.trace_rays(rays, algo, scale=FORM_SCALE, translation=tr, want_hits=True))
        s.close()
    return rays, out


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("kind,form,env", [("render",) + f for f in RENDER_FORMS] + [("trace",) + f for f in TRACE_FORMS],
                         ids=[f"render-{f}" for f, _ in RENDER_FORMS] + [f"trace-{f}" for f, _ in TRACE_FORMS])
def test_wide_kernel_forms_equal_the_default(default_outputs, kind, form, env):
    """Each render and trace form the environment switches select (tests/test_kernel_forms_gpu.py) on D = 200 at scale 3 with a large
    fractional translation: frames and hit maps, or trace colours and hit records, equal to the default form's for every combination."""
    rays, out = default_outputs
    tr = SCALES[FORM_SCALE]
    for storage, algo in COMBOS:
        s = gpu_scene("d200", storage, env)
        frames, traced = out[(storage, algo)]
        if kind == "render":
            for (o, l, fov), want in zip(wide_cameras("d200", FORM_SCALE, tr), frames):
                got = s.render(GW, GH, algo, cam(o, l, fov, GW, GH), scale=FORM_SCALE, translation=tr, want_hits=True)
                assert np.array_equal(got["rgb"], want["rgb"]) and np.array_equal(got["hits"], want["hits"]), (form, storage, algo, o)
        else:
            got = s.trace_rays(rays, algo, scale=FORM_SCALE, translation=tr, want_hits=True)
            assert np.array_equal(got["colour"], traced["colour"]) and np.array_equal(got["hits"], traced["hits"]), (form, storage, algo)
        s.close()
