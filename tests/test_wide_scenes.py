"""CPU tier: renders, traces, exact casts and the shadow horizon map on wide region tables (tests.common.WIDE_SCENES: D = 26 .. 1024,
negative min_coord, content far from region 0 and near both ends of the table, long runs of null regions) and at scales that are not
powers of two with fractional and large translations.  The product's traversal built for the host (tests/hostsim) against the oracle
bit for bit, the map's bound (no occupied-cluster test past a shadow ray's threshold) where its cells are wider than 8 voxels, and the
host build of cast_ray against the numpy cell-by-cell walk of tests/cast_ref.py."""
import ctypes as C

import numpy as np
import pytest

from tests import cast_ref as cr
from tests import horizon_sim as hs
from tests import surface_ref as sr
from tests.common import COMBOS, WIDE_SCENES, build_oracle, camera, horizon_grid, po, wide_scene

KIND = "orc"      # the oracle's C restatement: its region table is a calloc, so a wide table costs virtual memory only
FORMS = {"nested": 0, "fast": 3}     # sim_set_flat: vrm_core.cuh's nested loops; vrm_flat.cuh's state machine with its fast paths
F32 = np.float32
W, H = 64, 36
_SCENES = {}


def scene(name):
    if name not in _SCENES:
        _SCENES[name] = wide_scene(name)
    return _SCENES[name]


def table_box(name):
    """[L, H) in voxels of the table on every axis."""
    lo, hi = WIDE_SCENES[name][0]
    return 64 * lo, 64 * (hi + 1)


def centre(piece):
    return piece[0].mean(0)


def to_world(local, scale, translation):
    return (np.asarray(local, np.float64) / scale + np.asarray(translation, np.float64)).astype(F32)


def wide_cameras(name, scale=1, translation=(0.0, 0.0, 0.0)):
    """(origin, look_at, fov) in world units: inside the table over a piece, at the table's far corner looking at the farthest piece across
    the null regions, and outside the table at 10^3, 10^4 and 10^5 voxels with a field of view that frames a piece."""
    _, _, pieces = scene(name)
    L, Hb = table_box(name)
    c0, c1 = centre(pieces[0]), centre(pieces[-1])
    cams = [(c0 + (70.0, 90.0, 60.0), c0, 60.0)]
    corner = np.full(3, Hb - 3.5)
    far = max(pieces, key=lambda p: np.linalg.norm(centre(p) - corner))
    cams.append((corner, centre(far), float(np.degrees(2 * np.arctan(80.0 / np.linalg.norm(centre(far) - corner))))))
    for k, dist in enumerate((1e3, 1e4, 1e5)):
        u = np.array([(-1.0) ** k, 0.6, 0.45 * (-1.0) ** (k // 2)])
        u /= np.linalg.norm(u)
        tgt = centre(pieces[k % len(pieces)])
        out = np.where(u > 0, Hb, L) - tgt             # outside the table's box along u, then dist more
        org = tgt + u * (np.max(np.abs(out)) * 1.8 + dist)
        cams.append((org, tgt, float(np.degrees(2 * np.arctan(70.0 / np.linalg.norm(org - tgt))))))
    return [(tuple(to_world(o, scale, translation).tolist()), tuple(to_world(l, scale, translation).tolist()), fov) for o, l, fov in cams]


def wide_rays(name, n, seed, scale=1, translation=(0.0, 0.0, 0.0)):
    """World rays (m, 6): from 10^3 .. 10^5 voxels outside the table towards stored voxels (some deflected into misses), across the whole
    table from face to face through its null runs (half of them through a piece), and from origins whose table-relative coordinates are
    above 2^15 on an axis when the table is wide enough (else just outside its far faces)."""
    rng = np.random.default_rng(seed)
    _, _, pieces = scene(name)
    L, Hb = table_box(name)
    vox = np.concatenate([p[0] for p in pieces]).astype(np.float64)
    tgt = vox[rng.integers(0, len(vox), n)] + rng.uniform(0, 1, (n, 3))
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    org = tgt + u * ((Hb - L) * 1.8 + 10.0 ** rng.uniform(3, 5, (n, 1)))
    d = tgt - org + np.where(rng.random((n, 1)) < 0.25, rng.normal(0, 300, (n, 3)), 0.0)
    far = np.concatenate([org, d], 1)
    # face to face
    a = rng.integers(0, 3, n)
    org = rng.uniform(L, Hb, (n, 3))
    org[np.arange(n), a] = L - rng.uniform(1, 200, n)
    end = np.where(rng.random((n, 1)) < 0.5, tgt, rng.uniform(L, Hb, (n, 3)))
    end = end + (end - org) * 10.0
    cross = np.concatenate([org, end - org], 1)
    # table-relative coordinates above 2^15 (or beyond the far faces)
    org = tgt + rng.normal(0, 400, (n, 3))
    a = rng.integers(0, 3, n)
    org[np.arange(n), a] = np.maximum(L + 32768 + rng.uniform(1, 20000, n), Hb + rng.uniform(0.5, 3000, n)) if Hb - L <= 32768 else \
        L + rng.uniform(32768.5, Hb - L - 1, n)
    d = tgt - org + rng.normal(0, 30, (n, 3))
    high = np.concatenate([org, d], 1)
    rays = np.concatenate([far, cross, high])
    rays[:, 3:] /= np.linalg.norm(rays[:, 3:], axis=1, keepdims=True)
    return np.concatenate([to_world(rays[:, :3], scale, translation), rays[:, 3:].astype(F32)], 1)


@pytest.fixture
def lighting():
    """Restores the default light (unit (1, 1, 1)) and the state machine form on every library a test sets."""
    yield
    for kind in (KIND, "sim"):
        po.set_lighting(kind)
    po._lib("sim").sim_set_flat(1)
    hs.set_form(1)
    hs.set_lighting(po.unit_vector((1.0, 1.0, 1.0), KIND))


def set_light(direction):
    d = po.unit_vector(direction, KIND) if np.linalg.norm(direction) != 1.0 else np.asarray(direction, F32)
    for kind in (KIND, "sim"):
        po.set_lighting(kind, direction=d)
    hs.set_lighting(d)
    return d


# ---- the scenes and their horizon cells --------------------------------------------------------------------------------------------------

# (scene, light, cell width the map of that light must have)
CELLS = [("d26", (1.0, 1.0, 1.0), 8.0), ("d200", (1.0, 1.0, 1.0), 16.0), ("d200", (-0.3, -0.8, 0.5), 16.0), ("d200", (0.0, 1.0, 0.0), 8.0),
         ("d512", (0.0, 1.0, 0.0), 32.0), ("d512", (1.0, 1.0, 1.0), 32.0), ("d1024lo", (0.0, 0.0, -1.0), 64.0)]


@pytest.mark.parametrize("name", ["d26", "d200", "d512"])
def test_wide_tables_build_like_the_oracle(name):
    """Diameter and min_coord of each wide scene, every stored voxel and random misses looked up the same in the oracle and the host build,
    and the horizon cell width of horizon_setup restated (tests.common.horizon_grid) for the lights the map tests use."""
    xyz, rgb, _ = scene(name)
    lo, hi = WIDE_SCENES[name][0]
    L, Hb = table_box(name)
    q = np.concatenate([xyz, np.random.default_rng(3).integers(L - 70, Hb + 70, (20000, 3))]).astype(np.int32)
    for storage in ("vcs", "hashtable"):
        a, b = build_oracle(KIND, xyz, rgb, storage), build_oracle("sim", xyz, rgb, storage)
        assert a.info() == b.info() and (a.info()["diameter"], a.info()["min_coord"]) == (hi - lo + 1, lo)
        for x, y in zip(a.lookup(q), b.lookup(q)):
            assert np.array_equal(x, y)
        a.close()
    for sname, light, cell in CELLS:
        if sname == name:
            assert horizon_grid(po.unit_vector(light, KIND), hi - lo + 1)[0] == cell, (name, light)


def test_horizon_cells_wider_than_eight_voxels():
    """The map tests below reach cells of 16, 32 and 64 voxels; horizon_grid agrees with the sizes stated in kHorizonMaxCells' comment:
    the cell grows past 8 voxels from 157 regions on for a (1, 1, 1) light and from 256 regions on for an axis-aligned one."""
    for name, light, cell in CELLS:
        lo, hi = WIDE_SCENES[name][0]
        assert horizon_grid(po.unit_vector(light, KIND), hi - lo + 1)[0] == cell, (name, light)
    diag, axis = po.unit_vector((1.0, 1.0, 1.0), KIND), np.array([0.0, 1.0, 0.0], F32)
    assert horizon_grid(diag, 156)[0] == 8.0 and horizon_grid(diag, 157)[0] == 16.0
    assert horizon_grid(axis, 255)[0] == 8.0 and horizon_grid(axis, 256)[0] == 16.0


# ---- the horizon bound -------------------------------------------------------------------------------------------------------------------

def threshold_lights(rng):
    """Unit lights (float32) for the bound: random ones with every |component| >= 0.0625; ones with a component of exactly +-0.0625 and
    one float above it (whose normalised double is still >= 0.0625, so they get a map); axis-aligned; negative components."""
    out = []
    while len(out) < 4:
        v = rng.normal(size=3)
        u = v / np.linalg.norm(v)
        if np.all(np.abs(u) >= 0.07):
            out.append(po.unit_vector(tuple(v), KIND))
    for sign in (1.0, -1.0):
        for c in (F32(0.0625), np.nextafter(F32(0.0625), F32(1))):
            for z in np.linspace(0.2, 0.8, 2001, dtype=F32):
                y = F32(np.sqrt(np.float64(1.0) - np.float64(c) ** 2 - np.float64(z) ** 2))
                d = np.array([sign * c, y, -z], F32)
                if horizon_grid(d, 512) is not None:
                    out.append(d)
                    break
            else:
                raise AssertionError((sign, c))
    out += [np.array(v, F32) for v in ((0.0, 1.0, 0.0), (1.0, 0.0, 0.0), (0.0, 0.0, -1.0), (0.0, -1.0, 0.0))]
    out += [po.unit_vector(v, KIND) for v in ((-0.3, -0.8, 0.5), (0.3, 0.7, -0.65), (-1.0, 0.2, -0.4))]
    return out


def surface_rays(pieces, n, rng, light):
    """Rays from random points on the light's side of each piece towards its stored voxels: their hits (and shadow-ray starts) spread over
    every piece, near both ends of the table where the pieces lie there."""
    out = []
    for p in pieces:
        tgt = p[0][rng.integers(0, len(p[0]), n)].astype(np.float64) + 0.5
        org = tgt + rng.normal(size=(n, 3)) * 40.0 + np.asarray(light, np.float64) * 80.0
        d = tgt - org
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        out.append(np.concatenate([org, d], 1))
    return np.concatenate(out).astype(F32)


@pytest.mark.parametrize("algo", ["longestaxis", "original"])
@pytest.mark.parametrize("name", ["d200", "d512"])
def test_horizon_bound_on_wide_tables(lighting, name, algo):
    """hz_property on cells of 16 and 32 voxels: every shadow ray marched in full never finds an occupied cluster once it is past the threshold
    of its one map lookup, for random lights, lights at the 0.0625 component limit, axis-aligned lights and negative components."""
    rng = np.random.default_rng(7 if name == "d200" else 8)
    xyz, rgb, pieces = scene(name)
    D = WIDE_SCENES[name][0][1] - WIDE_SCENES[name][0][0] + 1
    b = hs.Scene(xyz, rgb)
    checked = passed = 0
    cells = []
    for d in threshold_lights(rng):
        grid = horizon_grid(d, D)
        assert grid is not None, (name, d)
        cells.append(grid[0])
        hs.set_lighting(d)
        res = b.property(surface_rays(pieces, 700, rng, d), algo)
        assert res is not None, (name, d)
        rays_n, bad, past, found = res
        assert bad == 0, (name, algo, d.tolist(), grid, res)
        checked += rays_n
        passed += past
    assert checked > 10000 and passed > checked // 10, (checked, passed)
    assert sum(c > 8 for c in cells) >= 7, cells          # (near-axis lights project the table narrowly: their cells stay smaller)


# ---- renders against the oracle, horizon on and off ------------------------------------------------------------------------------------

def check_render(name, storage, algo, scale=1, translation=(0.0, 0.0, 0.0), lights=((1.0, 1.0, 1.0),)):
    xyz, rgb, _ = scene(name)
    a, b = build_oracle(KIND, xyz, rgb, storage), hs.Scene(xyz, rgb, storage)
    hit_px = 0
    for light in lights:
        set_light(light)
        for o, l, fov in wide_cameras(name, scale, translation):
            cam = camera(o, l, fov, W, H, KIND)
            ref = a.render(cam, W, H, algo, scale=scale, translation=translation)
            off = b.render(cam, W, H, algo, scale=scale, translation=translation, horizon=False)
            on = b.render(cam, W, H, algo, scale=scale, translation=translation, horizon=True)
            tag = (name, storage, algo, scale, translation, light, o)
            for k in ("rgb", "hits"):
                assert np.array_equal(off[k], ref[k]), tag + (k, "map off")
                assert np.array_equal(on[k], ref[k]), tag + (k, "map on")
            assert np.all(on["counters"] <= off["counters"]), tag + (on["counters"], off["counters"])
            hit_px += int((ref["hits"][..., 3] != 0).sum())
    a.close()
    assert hit_px > len(lights) * W * H // 8, (name, hit_px)     # the cameras see the pieces


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("storage,algo", COMBOS)
@pytest.mark.parametrize("name", ["d26", "d200", "d512"])
def test_wide_renders_match_oracle(lighting, name, storage, algo, form):
    """RGB and hit maps bit for bit with the map on and off (cameras inside the table, at its far corner, and 10^3 .. 10^5 voxels out),
    and no more as-executed work with the map.  D = 26, 200 (map cells of 16 voxels) and 512 (32), lights diagonal, negative, axis."""
    hs.set_form(FORMS[form])
    check_render(name, storage, algo, lights=((1.0, 1.0, 1.0), (-0.3, -0.8, 0.5), (0.0, 1.0, 0.0)) if form == "fast" else ((1.0, 1.0, 1.0),))


# ---- traces against the oracle -----------------------------------------------------------------------------------------------------------

def check_traces(name, storage, algo, form, rays, scale=1, translation=(0.0, 0.0, 0.0), counters=True):
    xyz, rgb, _ = scene(name)
    po._lib("sim").sim_set_flat(FORMS[form])
    a, b = build_oracle(KIND, xyz, rgb, storage), build_oracle("sim", xyz, rgb, storage)
    ta = a.trace_rays(rays, algo, scale=scale, translation=translation, want_counters=counters)
    tb = b.trace_rays(rays, algo, scale=scale, translation=translation, want_counters=counters)
    a.close()
    b.close()
    for k in ("colour", "hits") + (("counters",) if counters else ()):
        assert np.array_equal(ta[k], tb[k]), (name, storage, algo, form, scale, translation, k,
                                              int((ta[k] != tb[k]).reshape(len(ta[k]), -1).any(1).sum()) if k != "counters" else ta[k])
    return ta


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("storage,algo", COMBOS)
@pytest.mark.parametrize("name", ["d26", "d200", "d512"])
def test_wide_traces_match_oracle(lighting, name, storage, algo, form):
    """Rays from far outside, face to face across the table through its null runs, and from table-relative coordinates above 2^15: colours,
    hit records and event counters of the nested form and of the state machine with its fast paths equal the oracle's."""
    rays = wide_rays(name, 1500, seed=len(name))
    ta = check_traces(name, storage, algo, form, rays)
    assert (ta["hits"][:, 3] != 0).sum() > 800


# ---- scales that are not powers of two, fractional and large translations ---------------------------------------------------------------

SCALED = [(3, (-40000.5, 1234.25, 60000.0)), (5, (0.3, -0.7, 0.1)), (12, (1024.75, -3.5, -20000.125)), (100, (-7.25, 50.5, 8.0))]


@pytest.mark.parametrize("scale,translation", SCALED, ids=[f"scale{s}" for s, _ in SCALED])
def test_wide_scaled_renders_and_traces_match_oracle(lighting, scale, translation):
    """D = 200 at scales 3, 5, 12 and 100 with fractional and large translations (cameras and rays placed to match): renders with the map on
    and off, and traces of both forms, both storages and both algorithms, against the oracle."""
    hs.set_form(3)
    rays = wide_rays("d200", 600, seed=scale, scale=scale, translation=translation)
    for storage, algo in COMBOS:
        check_render("d200", storage, algo, scale, translation)
        for form in FORMS:
            ta = check_traces("d200", storage, algo, form, rays, scale, translation)
            assert (ta["hits"][:, 3] != 0).sum() > 300


def test_d1024_trace_and_horizon_bound(lighting):
    """D = 1024 with content at x = -65472 and next to region 0 (min_coord -1023; the oracle's table is an 8 GiB virtual calloc, the host
    build's 4 GiB): a bounded ray set of both algorithms in the state machine against the oracle, and the map's bound on cells of 64 voxels."""
    xyz, rgb, pieces = scene("d1024lo")
    rays = wide_rays("d1024lo", 500, seed=4)
    for algo in ("longestaxis", "original"):
        ta = check_traces("d1024lo", "vcs", algo, "fast", rays)
        assert (ta["hits"][:, 3] != 0).sum() > 300
    b = hs.Scene(xyz, rgb)
    rng = np.random.default_rng(11)
    passed = 0
    for light in ((0.0, 0.0, -1.0), (1.0, 1.0, 1.0), (-0.3, -0.8, 0.5)):
        d = set_light(light)
        assert horizon_grid(d, 1024)[0] == 64.0
        for algo in ("longestaxis", "original"):
            res = b.property(surface_rays(pieces, 800, rng, d), algo)
            assert res is not None and res[1] == 0, (light, algo, res)
            passed += res[2]
    assert passed > 0


# ---- the 18-bit threshold clamps ---------------------------------------------------------------------------------------------------------

def test_threshold_is_clamped_not_wrapped(lighting):
    """horizon_threshold's value travels in bits 14..31 of the flag word.  Start points with a cell value (their map lookup) pushed so far that
    the computed threshold leaves [kHzMin, kHzNever] = [-131072, 131071] must give the clamp, and in-range values themselves, decoded
    from the word start_shadow wrote."""
    lib = hs.load()
    xyz, rgb, pieces = scene("d512")
    b = hs.Scene(xyz, rgb)
    L, Hb = table_box("d512")
    lo = WIDE_SCENES["d512"][0][0]
    rng = np.random.default_rng(5)
    for light in ((1.0, 1.0, 1.0), (-0.3, -0.8, 0.5), (0.0, 1.0, 0.0), (0.0, 0.0, -1.0)):
        d = set_light(light)
        grid = horizon_grid(d, 512)
        n = 400
        hit = np.concatenate([rng.uniform(L + 0.5, L + 70, (n // 2, 3)), rng.uniform(Hb - 70, Hb - 0.5, (n // 2, 3))])   # both ends
        reg = np.floor_divide(hit, 64).astype(np.int32)
        local = (hit - 64.0 * reg).astype(F32)
        for cell_value in (None, 1000000, 140000, -140000, -1000000, 0):
            for la in (0, 1):
                thr = np.zeros(n, np.int32)
                word = np.zeros(n, np.int32)
                computed = np.zeros(n, F32)
                rc = lib.hz_threshold_check(b.h, hs._p(np.ascontiguousarray(local)), hs._p(np.ascontiguousarray(reg)), C.c_uint64(n), int(la),
                                            C.c_int(0 if cell_value is None else 1), C.c_int32(cell_value or 0),
                                            hs._p(computed), hs._p(thr), hs._p(word))
                assert rc == 0, rc
                none = np.isnan(computed)        # no threshold axis (the original walk's x with n_x = 0)
                want = np.where(none | (computed >= 131071), 131071, np.where(computed <= -131072, -131072, np.nan_to_num(computed))).astype(np.int64)
                tag = (light, cell_value, la)
                assert np.array_equal(thr, want), tag
                assert np.array_equal(word, thr), tag
                if none.all():
                    continue
                if cell_value == 1000000:
                    assert (computed[~none] > 131071).any() and (thr[~none] == 131071).all(), tag
                elif cell_value == -1000000:
                    assert (computed[~none] < -131072).any() and (thr[~none] == -131072).any(), tag
                elif cell_value is None:
                    # the real map: an empty cell (kHorizonEmpty) clamps to kHzMin; every other value stays well inside the 18 bits,
                    # within a cell's reach of the table (|table-relative coordinate| < 65536), as the comment on horizon_threshold argues
                    real = ~none & (computed > -1e8)
                    assert real.any() and (np.abs(computed[real]) < 32768 + 400).all(), (tag, computed[real].min(), computed[real].max())
                    assert (thr[~none & ~real] == -131072).all(), tag
        assert grid[0] == 32.0 and lo == -300


# ---- exact casts ---------------------------------------------------------------------------------------------------------------------------

_CAST = {}


def cast_scene(name):
    if name not in _CAST:
        xyz, rgb, _ = scene(name)
        _CAST[name] = (cr.Stored(xyz, rgb), {s: cr.Sim(xyz, rgb, s) for s in ("vcs", "hashtable")})
    return _CAST[name]


def cast_cases(name, n, seed, scale=1, translation=(0.0, 0.0, 0.0)):
    """dict case -> (world rays, ranges or None) for the wide scene `name`.  The numpy walk steps cell by cell, so every interval that crosses
    the table's null runs is bounded to a few thousand cells: ranges that start in the null run before a piece and end inside or after it,
    ranges that end in the middle of a null run, and (D = 26 only) whole rays across the table."""
    rng = np.random.default_rng(seed)
    _, _, pieces = scene(name)
    L, Hb = table_box(name)
    vox = np.concatenate([p[0] for p in pieces]).astype(np.float64)
    tgt = vox[rng.integers(0, len(vox), n)] + rng.uniform(0, 1, (n, 3))
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    dist = (Hb - L) * 1.8 + 10.0 ** rng.uniform(3, 5, (n, 1))
    org = tgt + u * dist
    d = (tgt - org) / dist + np.where(rng.random((n, 1)) < 0.2, rng.normal(0, 0.004, (n, 3)), 0.0)
    t_hit = dist[:, 0]
    out = {}
    near = t_hit - rng.uniform(20, 1500, n)
    out["null_to_piece"] = (org, d, np.stack([near, near + rng.uniform(1, 2500, n)], 1))
    mid = t_hit - rng.uniform(400, 1500, n)
    out["ends_in_null"] = (org, d, np.stack([mid - rng.uniform(0, 800, n), mid], 1))
    # short intervals from the middle of the table: the start cell is found inside a long null run, far from region 0
    o2 = rng.uniform(L, Hb, (n, 3))
    d2 = tgt - o2
    d2 /= np.linalg.norm(d2, axis=1, keepdims=True)
    t2 = np.linalg.norm(tgt - o2, axis=1)
    s2 = np.maximum(t2 - rng.uniform(5, 1200, n), 0.0)
    out["inside_null"] = (o2, d2, np.stack([s2, s2 + rng.uniform(0, 2400, n)], 1))
    if Hb - L <= 2048:
        a = rng.integers(0, 3, n)
        o3 = rng.uniform(L, Hb, (n, 3))
        o3[np.arange(n), a] = L - rng.uniform(1, 5000, n)
        out["across"] = (o3, tgt - o3, None)
    res = {}
    for k, (o, dd, rg) in out.items():
        rays = np.concatenate([to_world(o, scale, translation), dd.astype(F32)], 1)
        res[k] = (rays, None if rg is None else (rg / scale).astype(F32))
    return res


WIDE_CASTS = [("d26", 1, (0.0, 0.0, 0.0)), ("d26", 3, (0.3, -0.7, 0.1)), ("d200", 1, (0.0, 0.0, 0.0)), ("d200", 5, (-40000.5, 1234.25, 60000.0)),
              ("d512", 1, (0.0, 0.0, 0.0)), ("d512", 12, (0.75, -1.25, 2.5)), ("d512", 100, (-7.25, 50.5, 8.0))]


@pytest.mark.parametrize("name,scale,translation", WIDE_CASTS, ids=[f"{n}-scale{s}" for n, s, _ in WIDE_CASTS])
def test_wide_casts_match_numpy_walk(name, scale, translation):
    """cast_ray's leaps over null regions and empty clusters, its start-cell search in a long null run and its entry into the table's box
    from far outside: both storages equal the cell-by-cell walk bit for bit."""
    st, sims = cast_scene(name)
    hits = 0
    for case, (rays, ranges) in cast_cases(name, 500, seed=scale + len(name), scale=scale, translation=translation).items():
        want = cr.cast_rays(st, rays, ranges, scale, translation)
        for storage, sim in sims.items():
            assert cr.same(sim.cast_rays(rays, ranges, scale, translation), want), (name, scale, case, storage)
        hits += int(want["hits"][:, 3].sum())
    assert hits > 400, hits


@pytest.mark.parametrize("scale", [1, 3, 5, 8, 12, 100])
def test_cast_depth_within_one_ulp_of_the_interval(scale):
    """The header's statement on ray intervals: an entered-cell hit's depth lies in [t_near, t_far] exactly at power-of-two scales, and within
    one ulp of it otherwise.  Intervals are cut a few ulps around the hit depths of full casts, so the edges are reached."""
    translation = (0.3, -0.7, 0.1) if scale % 2 else (0.0, 0.0, 0.0)
    st, sims = cast_scene("d200")
    sim = sims["vcs"]
    rays, ranges = cast_cases("d200", 600, seed=scale, scale=scale, translation=translation)["null_to_piece"]
    full = sim.cast_rays(rays, ranges, scale, translation)
    ent = (full["hits"][:, 3] != 0) & (full["face"] != 0)
    assert ent.sum() > 200
    r, d, t0, t1 = rays[ent], full["depth"][ent], ranges[ent, 0], ranges[ent, 1]
    outside = 0
    for k in (-2, -1, 0, 1, 2):
        edge = d.copy()
        for _ in range(abs(k)):
            edge = np.nextafter(edge, F32(np.inf if k > 0 else -np.inf))
        for rg in (np.stack([edge, t1], 1), np.stack([t0, edge], 1)):
            rg = np.ascontiguousarray(rg, F32)
            got = sim.cast_rays(r, rg, scale, translation)
            assert cr.same(got, cr.cast_rays(st, r, rg, scale, translation)), (scale, k)
            e = (got["hits"][:, 3] != 0) & (got["face"] != 0)
            dep, lo, hi = got["depth"][e], rg[e, 0], rg[e, 1]
            below, above = dep < lo, dep > hi
            if scale & (scale - 1) == 0:
                assert not below.any() and not above.any(), (scale, k)
            else:
                assert (dep[below] == np.nextafter(lo[below], F32(-np.inf))).all(), (scale, k)
                assert (dep[above] == np.nextafter(hi[above], F32(np.inf))).all(), (scale, k)
                outside += int(below.sum() + above.sum())
    if scale & (scale - 1):
        assert outside > 0, scale        # the one-ulp case is reached
    # the same depths equal the hit surfaces' for the same records
    want_d, _ = sr.rays(full["hits"][ent], r, scale, translation)
    assert np.array_equal(d, want_d)
