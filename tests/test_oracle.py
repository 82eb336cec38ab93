"""CPU tier: pins the oracle.  (1) The C restatement (oracle/vrm_oracle.c) against the committed golden fixtures, which
were produced by the UNMODIFIED reference built for the host; (2) when that reference build is present
(oracle/_ref/libvrm_ref_host.so), a live differential run of restatement vs reference."""
import os

import numpy as np
import pytest

from tests.common import COMBOS, GOLDEN_DIR, MINI_CAMERAS, PROBE_CAMERAS, build_oracle, camera, lookup_queries, po, scenes

W, H = 160, 90


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(GOLDEN_DIR, "reference_golden.npz"))


SCENES = {"probe": (scenes.probe_scene, 8, PROBE_CAMERAS), "mini": (scenes.mini_scene, 1, MINI_CAMERAS)}


@pytest.mark.parametrize("name", ["probe", "mini"])
@pytest.mark.parametrize("storage", ["hashtable", "vcs"])
def test_port_matches_golden(golden, name, storage):
    gen, scale, cams = SCENES[name]
    xyz, rgb = gen()
    po.set_lighting("orc")
    s = build_oracle("orc", xyz, rgb, storage)
    info = s.info()
    assert [info["diameter"], info["min_coord"], info["filled"]] == golden[f"{name}_{storage}_info"].tolist()
    val, ex = s.lookup(golden[f"{name}_queries"])
    assert np.array_equal(val, golden[f"{name}_{storage}_lookup"])
    assert np.array_equal(ex, golden[f"{name}_{storage}_exists"])
    for ci in range(len(cams)):
        cam = golden[f"{name}_cam{ci}"]
        for algo in ("original", "longestaxis"):
            r = s.render(cam, W, H, algo, scale=scale)
            assert np.array_equal(r["hits"], golden[f"{name}_{storage}_{algo}_cam{ci}_hits"]), (name, storage, algo, ci)
            assert np.array_equal(r["rgb"], golden[f"{name}_{storage}_{algo}_cam{ci}_rgb"]), (name, storage, algo, ci)


@pytest.mark.parametrize("tag,kw", [("point", dict(use_point=True, position=(60.0, 90.0, 80.0))), ("noshadow", dict(use_shadows=False))])
def test_port_lighting_variants_match_golden(golden, tag, kw):
    xyz, rgb = scenes.probe_scene()
    cam = golden["probe_cam1"]
    try:
        po.set_lighting("orc", **kw)
        for storage, algo in COMBOS:
            s = build_oracle("orc", xyz, rgb, storage)
            r = s.render(cam, W, H, algo, scale=8)
            assert np.array_equal(r["rgb"], golden[f"probe_{storage}_{algo}_{tag}_rgb"]), (storage, algo, tag)
    finally:
        po.set_lighting("orc")


def test_camera_restatement_matches_golden(golden):
    for ci, (o, l, fov) in enumerate(PROBE_CAMERAS):
        assert np.array_equal(camera(o, l, fov, W, H, "orc"), golden[f"probe_cam{ci}"])


def test_last_write_wins_and_partition_rules():
    """VoxelSceneCPU.cuh:16-46: floor-division regions, positive-mod local coordinates, last insert wins."""
    xyz = np.array([[0, 0, 0], [0, 0, 0], [-1, -1, -1], [-64, 63, 64], [-65, 0, 0], [-1, -1, -1]], np.int32)
    rgb = np.array([1, 2, 3, 4, 5, 6], np.uint32)
    for storage in ("hashtable", "vcs"):
        s = build_oracle("orc", xyz, rgb, storage)
        assert s.info() == dict(diameter=4, min_coord=-2, filled=4)
        val, _ = s.lookup(np.array([[0, 0, 0], [-1, -1, -1], [-64, 63, 64], [-65, 0, 0], [1, 0, 0], [500, 0, 0]], np.int32))
        assert val.tolist() == [2, 6, 4, 5, po.EMPTY, po.EMPTY]


def test_empty_scene_renders_background():
    s = build_oracle("orc", np.zeros((0, 3), np.int32), np.zeros(0, np.uint32), "vcs")
    assert s.info() == dict(diameter=1, min_coord=0, filled=0)
    r = s.render(camera(*PROBE_CAMERAS[0], 32, 18, "orc"), 32, 18, "original")
    assert not r["rgb"].any() and not r["hits"].any()


@pytest.mark.skipif(not po.available("refh"), reason="needs a build of the original project in oracle/_ref (oracle/Makefile, from a reference checkout that is not part of this repository)")
@pytest.mark.parametrize("storage,algo", COMBOS)
def test_port_matches_reference_live(storage, algo):
    """Differential run against the unmodified reference: RGB, hit map and per-pixel lookup counts must all agree."""
    po.set_lighting("orc")
    po.set_lighting("refh")
    xyz, rgb = scenes.probe_scene()
    a, b = build_oracle("refh", xyz, rgb, storage), build_oracle("orc", xyz, rgb, storage)
    assert a.info() == b.info()
    q = lookup_queries(xyz, 5000, seed=3)
    for x, y in zip(a.lookup(q), b.lookup(q)):
        assert np.array_equal(x, y)
    for o, l, fov in PROBE_CAMERAS:
        cam = camera(o, l, fov, 320, 180, "refh")
        ra = a.render(cam, 320, 180, algo, scale=8, want_counters=True, want_lookups=True)
        rb = b.render(cam, 320, 180, algo, scale=8, want_counters=True, want_lookups=True)
        for k in ("rgb", "hits", "counters", "lookups"):
            assert np.array_equal(ra[k], rb[k]), (storage, algo, k)
    rays = scenes.random_rays(20000, (40.0, 30.0, 45.0), seed=42)
    ta, tb = a.trace_rays(rays, algo), b.trace_rays(rays, algo)
    assert np.array_equal(ta["colour"], tb["colour"]) and np.array_equal(ta["hits"], tb["hits"])


@pytest.mark.skipif(not po.available("refh"), reason="needs a build of the original project in oracle/_ref (oracle/Makefile, from a reference checkout that is not part of this repository)")
def test_scene_generators_match_reference_generators():
    """scenes.hollow_cube / sphere_shell restate VoxelCube.cuh / VoxelSphere.cuh: compare through the lookup seam."""
    ref = po.OracleScene("refh")
    ref.add_cube(20, 10, -40, 12)
    ref.add_sphere(32, 32, 32, 20)
    ref.add_sphere(100, 40, 40, 30, checkered=True)
    ref.build("hashtable")
    parts = [scenes.hollow_cube(20, 10, -40, 12), scenes.sphere_shell(32, 32, 32, 20), scenes.sphere_shell(100, 40, 40, 30, checkered=True)]
    xyz = np.concatenate([p[0] for p in parts])
    rgb = np.concatenate([p[1] for p in parts])
    mine = build_oracle("orc", xyz, rgb, "hashtable")
    assert ref.info() == mine.info()
    g = np.stack(np.meshgrid(np.arange(0, 135, dtype=np.int32), np.arange(-5, 75, dtype=np.int32), np.arange(-56, 75, dtype=np.int32), indexing="ij"), -1).reshape(-1, 3)
    assert np.array_equal(ref.lookup(g)[0], mine.lookup(g)[0])
