"""GPU tier (pytest -m gpu): the CUDA path, called through the C ABI of libvrm_b200.so, against the oracle on the same
seeded inputs; against the committed golden fixtures; against the reference's own CUDA kernels rebuilt for sm_100a; and,
at BASELINE.json's full sizes, through size-independent properties.

Bar: BIT-EXACT hit maps, colours and lookups (integer / index work; the fp32 walk is canonical IEEE without contraction,
SURVEY.md §7 hard part 1).  Only the comparison with the reference's DEFAULT (-fmad=true) CUDA build is toleranced:
>= 99.9 % of pixels within 1 LSB per channel (BASELINE.json north_star)."""
import os

import numpy as np
import pytest

from tests.common import COMBOS, GOLDEN_DIR, MINI_CAMERAS, PROBE_CAMERAS, build_oracle, camera, lookup_queries, oracle_kind, po, scenes
from voxelraymarcher_b200 import api

pytestmark = pytest.mark.gpu


def build_product(xyz, rgb, storage):
    s = api.VoxelScene(0)
    # several chunks: insertion order across vrm_scene_add_voxels calls is part of the contract
    n = xyz.shape[0]
    cuts = [0, n // 3, n // 3, 2 * n // 3, n]
    for a, b in zip(cuts[:-1], cuts[1:]):
        s.add_voxels(xyz[a:b], rgb[a:b])
    s.generate_voxel_scene(storage)
    return s


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(GOLDEN_DIR, "reference_golden.npz"))


@pytest.fixture(scope="module")
def probe():
    return scenes.probe_scene()


@pytest.mark.parametrize("name", ["probe", "mini"])
@pytest.mark.parametrize("storage", ["hashtable", "vcs"])
def test_build_and_lookup_match_oracle(name, storage):
    xyz, rgb = scenes.probe_scene() if name == "probe" else scenes.mini_scene()
    kind = oracle_kind()
    ref = build_oracle(kind, xyz, rgb, storage)
    s = build_product(xyz, rgb, storage)
    info = s.info()
    assert dict(diameter=info["diameter"], min_coord=info["min_coord"], filled=info["filled"]) == ref.info()
    assert info["unique_voxels"] == len({tuple(v) for v in xyz.tolist()})
    q = lookup_queries(xyz, 50000, seed=11)
    val, ex = s.lookup(q)
    rval, rex = ref.lookup(q)
    assert np.array_equal(val, rval)
    assert np.array_equal(ex, rex)
    assert (val[: xyz.shape[0]] != api.EMPTY).all()      # every inserted voxel is found ...
    assert (val[xyz.shape[0]:] == api.EMPTY).sum() > 0    # ... and the random probes include real misses


@pytest.mark.parametrize("storage,algo", COMBOS)
def test_render_matches_oracle_probe(probe, storage, algo):
    xyz, rgb = probe
    kind = oracle_kind()
    po.set_lighting(kind)
    ref = build_oracle(kind, xyz, rgb, storage)
    s = build_product(xyz, rgb, storage)
    for (w, h) in ((640, 360), (333, 187)):           # second size: ragged tiles at the right / bottom edge
        for o, l, fov in PROBE_CAMERAS:
            cam = api.Camera(o, l, (0.0, 1.0, 0.0), fov, np.float32(w) / np.float32(h))
            got = s.render(w, h, algo, cam, scale=8, want_hits=True)
            want = ref.render(cam.data, w, h, algo, scale=8)
            assert np.array_equal(got["hits"], want["hits"]), (storage, algo, o, int((got["hits"] != want["hits"]).any(-1).sum()))
            assert np.array_equal(got["rgb"], want["rgb"]), (storage, algo, o)


@pytest.mark.parametrize("name", ["probe", "mini"])
@pytest.mark.parametrize("storage", ["hashtable", "vcs"])
def test_render_matches_golden(golden, name, storage):
    xyz, rgb = scenes.probe_scene() if name == "probe" else scenes.mini_scene()
    scale = 8 if name == "probe" else 1
    s = build_product(xyz, rgb, storage)
    info = s.info()
    assert [info["diameter"], info["min_coord"], info["filled"]] == golden[f"{name}_{storage}_info"].tolist()
    val, ex = s.lookup(golden[f"{name}_queries"])
    assert np.array_equal(val, golden[f"{name}_{storage}_lookup"]) and np.array_equal(ex, golden[f"{name}_{storage}_exists"])
    ncam = len(PROBE_CAMERAS) if name == "probe" else len(MINI_CAMERAS)
    for ci in range(ncam):
        for algo in ("original", "longestaxis"):
            got = s.render(160, 90, algo, golden[f"{name}_cam{ci}"], scale=scale, want_hits=True)
            assert np.array_equal(got["hits"], golden[f"{name}_{storage}_{algo}_cam{ci}_hits"]), (name, storage, algo, ci)
            assert np.array_equal(got["rgb"], golden[f"{name}_{storage}_{algo}_cam{ci}_rgb"]), (name, storage, algo, ci)


@pytest.mark.parametrize("tag,kw", [("point", dict(use_point_light=True, light_position=(60.0, 90.0, 80.0))), ("noshadow", dict(use_shadows=False))])
def test_lighting_variants_match_golden(golden, probe, tag, kw):
    xyz, rgb = probe
    for storage, algo in COMBOS:
        s = build_product(xyz, rgb, storage)
        s.setup_constant_values(**kw)
        got = s.render(160, 90, algo, golden["probe_cam1"], scale=8)
        assert np.array_equal(got["rgb"], golden[f"probe_{storage}_{algo}_{tag}_rgb"]), (storage, algo, tag)


@pytest.mark.parametrize("storage,algo", COMBOS)
def test_trace_rays_matches_oracle(storage, algo):
    """BASELINE.json config 5 at oracle-friendly size: incoherent rays + shadow rays in a sparse many-region scene."""
    kind = oracle_kind()
    po.set_lighting(kind)
    xyz, rgb = scenes.sparse_shells(256, 64, seed=7, fill_pct=50)
    ref = build_oracle(kind, xyz, rgb, storage)
    s = build_product(xyz, rgb, storage)
    rays = scenes.random_rays(200000, (130.0, 97.0, 121.0), seed=42)
    got = s.trace_rays(rays, algo, want_hits=True)
    want = ref.trace_rays(rays, algo)
    assert np.array_equal(got["hits"], want["hits"])
    assert np.array_equal(got["colour"], want["colour"])
    assert want["hits"][:, 3].sum() > 1000


@pytest.mark.parametrize("storage", ["hashtable", "vcs"])
def test_statistics_match_oracle_counters(probe, storage):
    """The event counts that feed the roofline's algorithmic bytes equal the oracle recorder's."""
    xyz, rgb = probe
    kind = oracle_kind()
    po.set_lighting(kind)
    ref = build_oracle(kind, xyz, rgb, storage)
    s = build_product(xyz, rgb, storage)
    s.set_statistics(True)
    cam = api.Camera(*PROBE_CAMERAS[1][:2], (0.0, 1.0, 0.0), PROBE_CAMERAS[1][2], np.float32(320) / np.float32(180))
    for algo in ("original", "longestaxis"):
        s.render(320, 180, algo, cam, scale=8)
        st = s.get_statistics()
        want = ref.render(cam.data, 320, 180, algo, scale=8, want_counters=True)["counters"]
        assert [st["exist_checks"], st["exist_false"], st["lookups"], st["lookup_hits"]] == [int(v) for v in want[:4]]
        assert st["rays"] == 320 * 180
        # the counters of the work as executed: the production kernels do not trace the shadow ray of a pixel that is black already
        # (a normal facing away from the light: colour * !shadow = 0 either way) -- same frame, fewer events
        frame = s.render(320, 180, algo, cam, scale=8)["rgb"]
        s.set_statistics(True, as_executed=True)
        frame2 = s.render(320, 180, algo, cam, scale=8)["rgb"]
        st2 = s.get_statistics()
        s.set_statistics(True)
        assert np.array_equal(frame, frame2)
        assert st2["rays"] == st["rays"] and st2["lookup_hits"] <= st["lookup_hits"] and 0 < st2["exist_checks"] < st["exist_checks"]


def test_edge_cases():
    # empty scene
    s = api.VoxelScene(0)
    s.generate_voxel_scene("vcs")
    assert s.info()["diameter"] == 1 and s.info()["filled"] == 0
    cam = api.Camera((6.0, 2.0, 6.0), (0.0, 0.0, -1.0))
    r = s.render(64, 36, "longestaxis", cam, want_hits=True)
    assert not r["rgb"].any() and not r["hits"].any()
    # state errors are reported, not ignored
    with pytest.raises(api.VrmError):
        s.generate_voxel_scene("vcs")
    with pytest.raises(api.VrmError):
        s.add_voxels(np.zeros((1, 3), np.int32), np.zeros(1, np.uint32))
    t = api.VoxelScene(0)
    with pytest.raises(api.VrmError):
        t.render(8, 8, "original", cam)
    # duplicates: last write wins, across chunk boundaries too; single-voxel regions; negative coordinates
    xyz = np.array([[0, 0, 0]] * 5 + [[-1, -1, -1], [63, 63, 63], [64, 64, 64], [-64, 0, 0], [-65, 0, 0], [0, 0, 0]], np.int32)
    rgb = np.arange(1, len(xyz) + 1, dtype=np.uint32)
    for storage in ("hashtable", "vcs"):
        u = api.VoxelScene(0)
        for i in range(len(xyz)):
            u.insert_voxel(*xyz[i].tolist(), int(rgb[i]))
        u.generate_voxel_scene(storage)
        ref = build_oracle("orc", xyz, rgb, storage)
        assert u.info()["unique_voxels"] == 6
        q = lookup_queries(xyz, 2000, seed=3)
        assert np.array_equal(u.lookup(q)[0], ref.lookup(q)[0])
        assert u.lookup(np.array([[0, 0, 0]], np.int32))[0][0] == len(xyz)


@pytest.mark.parametrize("storage,algo", COMBOS)
def test_matches_reference_cuda_kernels(probe, storage, algo):
    """The reference's OWN kernels rebuilt for sm_100a: -fmad=false build bit-exact; default -fmad=true build within
    the north star's tolerance (>= 99.9 % of pixels within 1 LSB per channel)."""
    if not po.available("refgx") or not po.available("refg"):
        pytest.skip("needs a build of the original project in oracle/_ref (oracle/Makefile, from a reference checkout that is not part of this repository)")
    xyz, rgb = probe
    w, h = 640, 360
    s = build_product(xyz, rgb, storage)
    cam = api.Camera(*PROBE_CAMERAS[0][:2], (0.0, 1.0, 0.0), 60.0, np.float32(w) / np.float32(h))
    got = s.render(w, h, algo, cam, scale=8, want_hits=True)
    po.set_lighting("refgx")
    ex = build_oracle("refgx", xyz, rgb, storage)
    want = ex.render(cam.data, w, h, algo, scale=8)
    assert np.array_equal(got["hits"], want["hits"])
    assert np.array_equal(got["rgb"], want["rgb"])
    po.set_lighting("refg")
    fm = build_oracle("refg", xyz, rgb, storage)
    loose = fm.render(cam.data, w, h, algo, scale=8, want_hits=False)
    close = (np.abs(got["rgb"].astype(np.int32) - loose["rgb"].astype(np.int32)) <= 1).all(-1).mean()
    assert close >= 0.999, close


def test_full_size_terrain_properties():
    """BASELINE.json config 3 (512^3 terrain, ~30 M voxels, 3840x2160): too big for the CPU oracle inside a test, so
    check size-independent properties: every inserted voxel is found with its colour; every reported hit voxel is a
    stored voxel; background pixels are black and hit-less; the render is deterministic; a views batch equals
    single renders; hashtable and VCS agree on the stored set."""
    import torch
    xyz, rgb = scenes.terrain(512, 1234)
    assert 25_000_000 < xyz.shape[0] < 36_000_000
    w, h = 3840, 2160
    cam = api.Camera((-96.0, 352.0, -96.0), (256.0, 64.0, 256.0), (0.0, 1.0, 0.0), 60.0, np.float32(w) / np.float32(h))
    rng = np.random.default_rng(5)
    sample = rng.choice(xyz.shape[0], 400000, replace=False)
    hitsets = {}
    r64 = xyz >> 6
    n_regions = np.unique(r64[:, 0] + 8 * r64[:, 1] + 64 * r64[:, 2]).size
    for storage in ("vcs", "hashtable"):
        s = api.VoxelScene(0)
        s.add_voxels(xyz, rgb)
        s.generate_voxel_scene(storage)
        info = s.info()
        assert (info["diameter"], info["min_coord"], info["filled"], info["unique_voxels"]) == (8, 0, n_regions, xyz.shape[0])
        val, ex = s.lookup(xyz[sample])
        assert np.array_equal(val, rgb[sample]) and ex.all()
        above = xyz[sample] + np.array([0, 400, 0], np.int32)     # far above the terrain: nothing stored
        assert (s.lookup(above)[0] == api.EMPTY).all()
        for algo in ("original", "longestaxis"):
            a = s.render(w, h, algo, cam, want_hits=True)
            b = s.render(w, h, algo, cam, want_hits=True)
            assert np.array_equal(a["rgb"], b["rgb"]) and np.array_equal(a["hits"], b["hits"])
            hit = a["hits"][..., 3] == 1
            assert 0.3 < hit.mean() < 1.0
            assert not a["rgb"][~hit].any()
            coords = a["hits"][hit][:, :3]
            pick = rng.choice(coords.shape[0], 300000, replace=False)
            assert (s.lookup(coords[pick])[0] != api.EMPTY).all()
            hitsets[(storage, algo)] = a["hits"]
        # a batch of views in one launch equals the single renders
        cams = [cam, api.Camera((600.0, 300.0, 620.0), (256.0, 64.0, 256.0), (0.0, 1.0, 0.0), 60.0, np.float32(640) / np.float32(360))]
        cams[0] = api.Camera((-96.0, 352.0, -96.0), (256.0, 64.0, 256.0), (0.0, 1.0, 0.0), 60.0, np.float32(640) / np.float32(360))
        out = torch.zeros((2, 360, 640, 3), dtype=torch.uint8, device="cuda:0")
        s.render_views_device(640, 360, "longestaxis", cams, out.data_ptr())
        s.synchronize()
        for i in range(2):
            single = s.render(640, 360, "longestaxis", cams[i])
            assert np.array_equal(out[i].cpu().numpy(), single["rgb"])
        s.close()
    # hashtable never skips clusters, VCS does: images may legitimately differ in a few pixels (SURVEY.md §7 hard part 2)
    for algo in ("original", "longestaxis"):
        differ = (hitsets[("vcs", algo)] != hitsets[("hashtable", algo)]).any(-1).mean()
        print(f"hashtable vs vcs hit maps differ on {differ:.2e} of the pixels ({algo})")
        assert differ < 0.05, differ


@pytest.mark.timeout(300)
@pytest.mark.parametrize("storage,algo", COMBOS)
def test_axis_aligned_rays_terminate_and_match(probe, storage, algo):
    """Exactly-zero direction components: inf / NaN in the reference's unguarded divisions.  The kernels must terminate
    (the reference's own CUDA kernels would spin on a NaN position) and agree with the reference's HOST build."""
    from tests.test_hostsim import axis_aligned_rays
    xyz, rgb = probe
    kind = oracle_kind()
    po.set_lighting(kind)
    ref = build_oracle(kind, xyz, rgb, storage)
    s = build_product(xyz, rgb, storage)
    rays = axis_aligned_rays()
    got = s.trace_rays(rays, algo, want_hits=True)
    want = ref.trace_rays(rays, algo, threads=1)
    assert np.array_equal(got["colour"], want["colour"])
    assert np.array_equal(got["hits"], want["hits"])


def test_pinned_host_buffer_is_written_directly(probe):
    """vrm_render into page-locked memory (zero-copy stores from the kernel) equals the pageable path (device framebuffer +
    copy), for an aligned and for a ragged resolution, hits included."""
    import torch
    xyz, rgb = probe
    s = build_product(xyz, rgb, "vcs")
    for (w, h) in ((640, 360), (333, 187)):
        cam = api.Camera((14.0, 9.0, 12.0), (4.0, 3.0, 2.0), (0.0, 1.0, 0.0), 60.0, np.float32(w) / np.float32(h))
        want = s.render(w, h, "longestaxis", cam, scale=8, want_hits=True)
        pinned = torch.zeros((h, w, 3), dtype=torch.uint8).pin_memory()
        got = s.render(w, h, "longestaxis", cam, scale=8, rgb_out=pinned.numpy())
        assert np.array_equal(pinned.numpy(), want["rgb"])
        assert got["rgb"] is not None and want["hits"][..., 3].sum() > 0


@pytest.mark.parametrize("w,h", [(250, 141), (33, 5), (7, 3), (1, 1), (644, 362)])
def test_device_frames_at_ragged_resolutions_equal_host_frames(probe, w, h):
    """The fused kernel has two store forms with their own pixel-to-thread layout -- per-warp stores for a frame in the GPU's own memory,
    CTA-staged rows for a frame elsewhere (here: the handle's page-locked staging frame behind a pageable buffer).  Both must give the
    same frame at sizes that are no multiple of a tile or a CTA, for a single view and for a 3-view batch."""
    import torch
    xyz, rgb = probe
    s = build_product(xyz, rgb, "vcs")
    cams = [api.Camera((14.0 - 2.0 * v, 9.0, 12.0 + v), (4.0, 3.0, 2.0), (0.0, 1.0, 0.0), 60.0, np.float32(w) / np.float32(h)) for v in range(3)]
    want = [s.render(w, h, "longestaxis", c, scale=8)["rgb"] for c in cams]
    one = torch.full((h, w, 3), 7, dtype=torch.uint8, device="cuda:0")
    s.render_device(w, h, "longestaxis", cams[0], one.data_ptr(), scale=8)
    batch = torch.full((3, h, w, 3), 7, dtype=torch.uint8, device="cuda:0")
    s.render_views_device(w, h, "longestaxis", cams, batch.data_ptr(), scale=8)
    s.synchronize()
    assert np.array_equal(one.cpu().numpy(), want[0])
    for v in range(3):
        assert np.array_equal(batch[v].cpu().numpy(), want[v]), v
    s.close()


@pytest.mark.parametrize("storage,algo", COMBOS)
def test_remote_frame_rows_as_bulk_copies_equal_plain_stores(probe, storage, algo, monkeypatch):
    """A frame outside the GPU's own memory (here: page-locked host memory) leaves the CTA as bulk async copies (cp.async.bulk) when every
    96-byte row segment is 16-byte aligned, else as ordinary stores: both forms, at an aligned width, at a width whose rows are only
    4-byte aligned (W * 3 % 16 != 0) and through a frame base that is only 4-byte aligned, must equal the device-frame render."""
    import torch
    xyz, rgb = probe
    frames = {}
    for bulk in ("1", "0"):
        monkeypatch.setenv("VRM_BULK_STORE", bulk)   # read at vrm_scene_create
        s = build_product(xyz, rgb, storage)
        for (w, h, off) in ((640, 360, 0), (644, 360, 0), (640, 360, 4)):
            cam = api.Camera((14.0, 9.0, 12.0), (4.0, 3.0, 2.0), (0.0, 1.0, 0.0), 60.0, np.float32(w) / np.float32(h))
            dev = torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda:0")
            s.render_device(w, h, algo, cam, dev.data_ptr(), scale=8)
            s.synchronize()
            pinned = torch.zeros(h * w * 3 + 16, dtype=torch.uint8).pin_memory()
            view = pinned.numpy()[off:off + h * w * 3].reshape(h, w, 3)
            s.render(w, h, algo, cam, scale=8, rgb_out=view)
            assert np.array_equal(view, dev.cpu().numpy()), (bulk, w, h, off)
            assert view.any()
            frames[(bulk, w, off)] = view.copy()
        s.close()
    for (bulk, w, off), f in frames.items():
        assert np.array_equal(f, frames[("1", w, off)])


@pytest.mark.timeout(600)
@pytest.mark.parametrize("algo", ["original", "longestaxis"])
def test_crawl_fast_forward_is_bit_exact(algo):
    """Rays stuck on a cluster face (the reference advances them by EPSILON per iteration, ~5e7 iterations here): the
    kernels fast-forward the crawl and must return the same colours, hit voxels and event counters."""
    from tests.test_hostsim import crawl_scene_and_rays
    xyz, rgb, rays = crawl_scene_and_rays()
    kind = oracle_kind()
    po.set_lighting(kind)
    ref = build_oracle(kind, xyz, rgb, "vcs")
    s = build_product(xyz, rgb, "vcs")
    s.set_statistics(True)
    got = s.trace_rays(rays, algo, want_hits=True)
    st = s.get_statistics()
    want = ref.trace_rays(rays, algo, want_counters=True)
    assert np.array_equal(got["colour"], want["colour"])
    assert np.array_equal(got["hits"], want["hits"])
    assert [st["exist_checks"], st["exist_false"], st["lookups"], st["lookup_hits"]] == [int(v) for v in want["counters"][:4]]
    assert st["crawl_skipped"] > 10_000_000


@pytest.mark.parametrize("storage", ["vcs", "hashtable"])
@pytest.mark.parametrize("kind,kw", [("terrain", dict(size=192, seed=1234)), ("terrain", dict(size=96, seed=5, max_height=40)),
                                      ("shells", dict(size=256, cell=64, seed=7, fill_pct=50)), ("shells", dict(size=192, cell=32, seed=11, fill_pct=35))])
def test_gpu_scene_generators_match_host_generators(kind, kw, storage):
    """vrm_scene_generate_* put the same voxel set with the same colours into the staging list as scenes.terrain /
    scenes.sparse_shells: same structure geometry, every host-generated voxel found with its colour, same voxel count
    (so nothing extra), and a rendered frame that is bit-identical to the one of the host-generated scene."""
    xyz, rgb = scenes.terrain(**kw) if kind == "terrain" else scenes.sparse_shells(**kw)
    host = api.VoxelScene(0)
    host.add_voxels(xyz, rgb)
    host.generate_voxel_scene(storage)
    dev = api.VoxelScene(0)
    n = dev.generate_terrain(kw["size"], kw["seed"], kw.get("max_height", 0)) if kind == "terrain" else dev.generate_sparse_shells(kw["size"], kw["cell"], kw["seed"], kw["fill_pct"])
    assert n == xyz.shape[0]
    dev.generate_voxel_scene(storage)
    ih, idv = host.info(), dev.info()
    for k in ("diameter", "min_coord", "filled", "unique_voxels"):
        assert ih[k] == idv[k], k
    col, exists = dev.lookup(xyz)
    assert np.array_equal(col, rgb)
    q = lookup_queries(xyz, 20000, seed=3)
    a, b = host.lookup(q), dev.lookup(q)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    size = kw["size"]
    cam = api.Camera((-0.2 * size, 0.7 * size, -0.19 * size), (0.5 * size, 0.12 * size, 0.5 * size), (0.0, 1.0, 0.0), 60.0, np.float32(320) / np.float32(180))
    for algo in ("original", "longestaxis"):
        ra, rb = host.render(320, 180, algo, cam, want_hits=True), dev.render(320, 180, algo, cam, want_hits=True)
        assert np.array_equal(ra["rgb"], rb["rgb"]) and np.array_equal(ra["hits"], rb["hits"])
        assert int(ra["hits"][..., 3].sum()) > 1000
    host.close()
    dev.close()


def test_streaming_multi_view_render_equals_single_renders(probe, monkeypatch):
    """vrm_render_views (camera orbit into host frames): pageable frames go through double-buffered device batches (forced to
    2 views per batch here, so 7 views = 4 batches exercise the buffer hand-over), pinned frames are written directly; both must
    equal the single-frame renders bit for bit."""
    import torch
    xyz, rgb = probe
    w, h = 256, 144
    monkeypatch.setenv("VRM_VIEW_BATCH_BYTES", str(2 * w * h * 3))
    s = api.VoxelScene(0)
    s.add_voxels(xyz, rgb)
    s.generate_voxel_scene("vcs")
    cams = []
    for v in range(7):
        ang = 2.0 * np.pi * (v + 0.31) / 7
        cams.append(api.Camera((6.0 + 9.0 * np.cos(ang), 3.0 + 0.3 * v, 6.0 + 9.0 * np.sin(ang)), (6.0, 2.0, 2.0), (0.0, 1.0, 0.0), 60.0, np.float32(w) / np.float32(h)))
    for algo in ("longestaxis", "original"):
        singles = np.stack([s.render(w, h, algo, c, scale=8)["rgb"] for c in cams])
        assert singles.any()
        pageable = s.render_views(w, h, algo, cams, scale=8)
        assert np.array_equal(pageable["rgb"], singles)
        pinned = torch.zeros((7, h, w, 3), dtype=torch.uint8).pin_memory()
        got = s.render_views(w, h, algo, cams, scale=8, rgb_out=pinned.numpy())
        assert np.array_equal(got["rgb"], singles)
    s.close()


@pytest.mark.parametrize("storage,algo", COMBOS)
@pytest.mark.parametrize("w,h", [(250, 141), (33, 5), (7, 3), (1, 1)])
def test_ragged_resolutions_match_oracle(probe, storage, algo, w, h):
    """Image sizes that are not multiples of the 8x4 warp tile / 32x4 CTA (lanes and warps without a pixel take part in the
    warp-cooperative state machine; rows that are not 4-byte aligned take the per-pixel store path)."""
    xyz, rgb = probe
    kind = oracle_kind()
    po.set_lighting(kind)
    s = build_product(xyz, rgb, storage)
    ref = build_oracle(kind, xyz, rgb, storage)
    cam = camera((6.0, 2.0, 6.0), (0.0, 0.0, -1.0), 60.0, w, h, kind)
    got = s.render(w, h, algo, cam, scale=8, want_hits=True)
    want = ref.render(cam, w, h, algo, scale=8)
    assert np.array_equal(got["hits"], want["hits"])
    assert np.array_equal(got["rgb"], want["rgb"])
    s.close()


def test_scene_generator_argument_errors():
    s = api.VoxelScene(0)
    for bad in (dict(size=1), dict(size=5000)):
        with pytest.raises(api.VrmError):
            s.generate_terrain(bad["size"], 1)
    for size, cell in ((100, 64), (64, 4), (1024, 512)):
        with pytest.raises(api.VrmError):
            s.generate_sparse_shells(size, cell, 7, 35)
    assert s.generate_sparse_shells(128, 64, 7, 0) == 0          # nothing kept: an empty but valid scene
    s.generate_voxel_scene("vcs")
    with pytest.raises(api.VrmError):
        s.generate_terrain(64, 1)                                 # already built
    s.close()


def test_region_face_pingpong_and_tie_fast_forwards_are_bit_exact():
    """The two further forms of the reference's EPSILON crawl (tests/test_hostsim.py has the scenes): rays hopping across a region
    face twice per cycle (pingpong_skip) and crawl steps that are exact rounding ties (crawl_skip).  Oracle = millions of
    iterations; the kernels fast-forward them and must return the same colours, hit voxels and event counters."""
    from tests.test_hostsim import pingpong_scene_and_rays
    kind = oracle_kind()
    po.set_lighting(kind)
    xyz, rgb, rays = pingpong_scene_and_rays()
    s, ref = build_product(xyz, rgb, "vcs"), build_oracle(kind, xyz, rgb, "vcs")
    s.set_statistics(True)
    got, want = s.trace_rays(rays, "longestaxis", want_hits=True), ref.trace_rays(rays, "longestaxis", want_counters=True)
    st = s.get_statistics()
    assert np.array_equal(got["colour"], want["colour"]) and np.array_equal(got["hits"], want["hits"])
    assert (st["exist_checks"], st["exist_false"], st["lookups"]) == tuple(int(v) for v in want["counters"][:3])
    assert st["crawl_skipped"] > 0.9 * st["exist_checks"] > 4_000_000
    s.close()
    ys, zs = np.meshgrid(np.arange(0, 64, dtype=np.int32), np.arange(0, 64, dtype=np.int32), indexing="ij")
    xyz = np.stack([np.full(ys.size, 62, np.int32), ys.ravel(), zs.ravel()], 1)
    rgb = np.full(xyz.shape[0], 0x80C0F0, np.uint32)
    d = (0.848770142, -0.0162127428, -0.528513312)
    rays = np.array([[17.0, 48.02, 46.0, *d], [17.000002, 48.02, 46.0, *d], [9.0, 48.02, 46.0, *d], [33.0, 48.02, 46.0, *d]], np.float32)
    s, ref = build_product(xyz, rgb, "vcs"), build_oracle(kind, xyz, rgb, "vcs")
    s.set_statistics(True)
    for algo in ("original", "longestaxis"):
        got, want = s.trace_rays(rays, algo, want_hits=True), ref.trace_rays(rays, algo, want_counters=True)
        st = s.get_statistics()
        assert np.array_equal(got["colour"], want["colour"]) and np.array_equal(got["hits"], want["hits"]), algo
        assert (st["exist_checks"], st["exist_false"], st["lookups"]) == tuple(int(v) for v in want["counters"][:3]), algo
        if algo == "original":
            assert st["crawl_skipped"] > 0.9 * st["exist_checks"] > 250_000
    s.close()


@pytest.mark.parametrize("storage", ["vcs", "hashtable"])
def test_gpu_reference_generators_match_host_in_insertion_order(storage):
    """vrm_scene_generate_cube / _sphere = the reference's VoxelCube / VoxelSphere generators (scenes.hollow_cube / sphere_shell,
    which tests/test_oracle.py pins to the reference's functions).  The shapes overlap each other and a cube's faces overlap on
    its edges, so the built scenes only agree if the GPU generators also reproduce the INSERTION ORDER (last insert wins)."""
    parts = [("sphere", (40, 40, 40, 20, False)), ("cube", (44, 36, 52, 14)), ("sphere", (50, 44, 40, 17, True)), ("cube", (40, 40, 40, 9)),
             ("cube", (-30, 5, -70, 6)), ("sphere", (120, 70, 64, 30, True))]
    host, dev = api.VoxelScene(0), api.VoxelScene(0)
    total = 0
    for kind, args in parts:
        xyz, rgb = scenes.hollow_cube(*args) if kind == "cube" else scenes.sphere_shell(*args[:4], checkered=args[4])
        host.add_voxels(xyz, rgb)
        n = dev.generate_cube(*args) if kind == "cube" else dev.generate_sphere(*args)
        assert n == xyz.shape[0], (kind, args)
        total += n
    host.generate_voxel_scene(storage)
    dev.generate_voxel_scene(storage)
    ih, idv = host.info(), dev.info()
    for k in ("diameter", "min_coord", "filled", "unique_voxels"):
        assert ih[k] == idv[k], k
    assert ih["unique_voxels"] < total          # the overlaps are real
    allxyz = np.concatenate([(scenes.hollow_cube(*a) if k == "cube" else scenes.sphere_shell(*a[:4], checkered=a[4]))[0] for k, a in parts])
    q = lookup_queries(allxyz, 20000, seed=9)
    a, b = host.lookup(q), dev.lookup(q)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    with pytest.raises(api.VrmError):
        api.VoxelScene(0).generate_sphere(5, 40, 40, 20)          # centre closer to the origin than the radius: the reference's unsigned bounds wrap
    host.close()
    dev.close()


def test_full_defer_queue_falls_back_to_crawling(monkeypatch):
    """Rays that cannot be parked (queue of 3 slots, 12 ping-pong rays) crawl on in their kernel like the reference: same
    colours, hit voxels and counters, just slower."""
    from tests.test_hostsim import pingpong_scene_and_rays
    monkeypatch.setenv("VRM_DEFER_CAPACITY", "3")
    kind = oracle_kind()
    po.set_lighting(kind)
    xyz, rgb, rays = pingpong_scene_and_rays()
    s, ref = build_product(xyz, rgb, "vcs"), build_oracle(kind, xyz, rgb, "vcs")
    s.set_statistics(True)
    got, want = s.trace_rays(rays, "longestaxis", want_hits=True), ref.trace_rays(rays, "longestaxis", want_counters=True)
    st = s.get_statistics()
    assert np.array_equal(got["colour"], want["colour"]) and np.array_equal(got["hits"], want["hits"])
    assert (st["exist_checks"], st["exist_false"], st["lookups"]) == tuple(int(v) for v in want["counters"][:3])
    assert 0 < st["crawl_skipped"] < 0.6 * st["exist_checks"]      # three rays were fast-forwarded, nine crawled
    s.close()


def test_strided_view_batch_fills_interleaved_slots(probe):
    """vrm_render_views_device_strided: two "ranks" render the odd and the even views of a 5-view batch into one shared frame buffer
    (view_stride 2, starting at their own slot); the buffer must equal the single-frame renders, hit maps included."""
    import torch
    xyz, rgb = probe
    w, h = 160, 90
    s = build_product(xyz, rgb, "vcs")
    cams = [api.Camera((6.0 + 0.7 * v, 2.0 + 0.2 * v, 6.0 - 0.4 * v), (0.0, 0.0, -1.0), (0.0, 1.0, 0.0), 60.0, np.float32(w) / np.float32(h)) for v in range(5)]
    for algo in ("longestaxis", "original"):
        frames = torch.zeros((5, h, w, 3), dtype=torch.uint8, device="cuda:0")
        hits = torch.zeros((5, h, w, 4), dtype=torch.int32, device="cuda:0")
        for rank in range(2):
            mine = range(rank, 5, 2)
            s.render_views_device(w, h, algo, [cams[i] for i in mine], frames[rank].data_ptr(), hits[rank].data_ptr(), scale=8, view_stride=2)
        s.synchronize()
        for v in range(5):
            one = s.render(w, h, algo, cams[v], scale=8, want_hits=True)
            assert np.array_equal(frames[v].cpu().numpy(), one["rgb"]), (algo, v)
            assert np.array_equal(hits[v].cpu().numpy(), one["hits"]), (algo, v)
    s.close()


@pytest.mark.parametrize("algo", ["original", "longestaxis"])
def test_rays_starting_on_power_of_two_coordinates(algo):
    """The crawl_skip regression of tests/test_hostsim.py (an axis on a cluster face at local 16.0 is not stuck) through the kernels."""
    kind = oracle_kind()
    po.set_lighting(kind)
    xyz, rgb = scenes.terrain(160, 77)
    s, ref = build_product(xyz, rgb, "vcs"), build_oracle(kind, xyz, rgb, "vcs")
    rays = scenes.random_rays(20000, (80.0, 150.0, 80.0), seed=101)
    s.set_statistics(True)
    got, want = s.trace_rays(rays, algo, want_hits=True), ref.trace_rays(rays, algo, want_counters=True)
    st = s.get_statistics()
    assert np.array_equal(got["colour"], want["colour"]) and np.array_equal(got["hits"], want["hits"])
    assert (st["exist_checks"], st["exist_false"], st["lookups"]) == tuple(int(v) for v in want["counters"][:3])
    s.close()


@pytest.mark.parametrize("storage", ["vcs", "hashtable"])
def test_lookups_with_a_coordinate_of_64_are_empty(storage):
    """tests/test_hostsim.py coordinate64_rays through the kernels: rays rebased onto exactly 64.0 test voxels with a coordinate of 64,
    which match nothing in the reference.  (These exact rays cannot be had from a camera: the render kernels' source is covered by
    its host compile in tests/test_hostsim.py for this case.)"""
    from tests.test_hostsim import coordinate64_rays
    po.set_lighting("orc")
    xyz, rgb = scenes.probe_scene()
    s, ref = build_product(xyz, rgb, storage), build_oracle("orc", xyz, rgb, storage)
    rays = coordinate64_rays()
    got, want = s.trace_rays(rays, "longestaxis", scale=8, want_hits=True), ref.trace_rays(rays, "longestaxis", scale=8)
    assert not want["hits"][:, 3].any()
    assert np.array_equal(got["colour"], want["colour"]) and np.array_equal(got["hits"], want["hits"])
    s.close()


@pytest.mark.parametrize("storage,algo", COMBOS)
def test_scene_translation_matches_oracle(probe, storage, algo):
    """A non-zero VoxelSceneInfo translation (the reference's main always passes zero; its routines and this ABI take any) through
    the render and the trace kernels."""
    xyz, rgb = probe
    kind = oracle_kind()
    po.set_lighting(kind)
    ref, s = build_oracle(kind, xyz, rgb, storage), build_product(xyz, rgb, storage)
    o, l, fov = PROBE_CAMERAS[1]
    cam = api.Camera(o, l, (0.0, 1.0, 0.0), fov, np.float32(320) / np.float32(180))
    for tr in ((3.5, -2.25, 7.0), (-0.3, 0.7, 0.1)):
        got = s.render(320, 180, algo, cam, scale=8, translation=tr, want_hits=True)
        want = ref.render(cam.data, 320, 180, algo, scale=8, translation=tr)
        assert (want["hits"][..., 3] != 0).sum() > 4000
        assert np.array_equal(got["hits"], want["hits"]) and np.array_equal(got["rgb"], want["rgb"]), (storage, algo, tr)
        rays = scenes.random_rays(20000, (o[0] + 0.25, o[1], o[2]), seed=77)
        gt, wt = s.trace_rays(rays, algo, scale=8, translation=tr, want_hits=True), ref.trace_rays(rays, algo, scale=8, translation=tr)
        assert np.array_equal(gt["colour"], wt["colour"]) and np.array_equal(gt["hits"], wt["hits"]), (storage, algo, tr)
    s.close()


@pytest.mark.parametrize("storage", ["vcs", "hashtable"])
def test_device_pointer_entry_points_on_a_caller_stream(probe, storage):
    """vrm_scene_add_voxels_device / vrm_render_device / vrm_trace_rays_device on the caller's stream (the path a framework with its
    own device buffers takes, and the one bench.py times): same structure and same bytes as the host-buffer entry points; the opt-in
    L2 access-policy window changes nothing but cache behaviour."""
    import torch
    xyz, rgb = probe
    host = build_product(xyz, rgb, storage)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_xyz = torch.from_numpy(np.ascontiguousarray(xyz, np.int32)).cuda()
        d_rgb = torch.from_numpy(np.ascontiguousarray(rgb, np.uint32).view(np.int32)).cuda()
        s = api.VoxelScene(0)
        s.set_stream(stream.cuda_stream)
        half = len(rgb) // 2      # two chunks: staging keeps the insertion order across calls
        s.add_voxels_device(d_xyz.data_ptr(), d_rgb.data_ptr(), half)
        s.add_voxels_device(d_xyz[half:].data_ptr(), d_rgb[half:].data_ptr(), len(rgb) - half)
        s.generate_voxel_scene(storage)
        assert s.info() == host.info()
        o, l, fov = PROBE_CAMERAS[1]
        cam = api.Camera(o, l, (0.0, 1.0, 0.0), fov, np.float32(320) / np.float32(180))
        rays = scenes.random_rays(20000, o, seed=3)
        d_rays = torch.from_numpy(rays).cuda()
        for algo in ("longestaxis", "original"):
            want = host.render(320, 180, algo, cam, scale=8, want_hits=True)
            wt = host.trace_rays(rays, algo, scale=8, want_hits=True)
            for l2 in (False, True):
                s.set_l2_persistence(l2)
                fb = torch.zeros(180, 320, 3, dtype=torch.uint8, device="cuda")
                hits = torch.zeros(180, 320, 4, dtype=torch.int32, device="cuda")
                s.render_device(320, 180, algo, cam, fb.data_ptr(), hits.data_ptr(), scale=8)
                colour = torch.zeros(len(rays), dtype=torch.int32, device="cuda")
                rh = torch.zeros(len(rays), 4, dtype=torch.int32, device="cuda")
                s.trace_rays_device(d_rays.data_ptr(), len(rays), algo, colour.data_ptr(), rh.data_ptr(), scale=8)
                stream.synchronize()   # the calls are asynchronous on the caller's stream
                assert np.array_equal(fb.cpu().numpy(), want["rgb"]) and np.array_equal(hits.cpu().numpy(), want["hits"]), (storage, algo, l2)
                assert np.array_equal(colour.cpu().numpy().view(np.uint32), wt["colour"]) and np.array_equal(rh.cpu().numpy(), wt["hits"]), (storage, algo, l2)
        s.reset_stream()
        got = s.render(320, 180, "longestaxis", cam, scale=8)
        assert np.array_equal(got["rgb"], host.render(320, 180, "longestaxis", cam, scale=8)["rgb"])
    s.close(); host.close()


REGION_CORNER_CAMERAS = [((16.0, 8.0, 0.0), (15.9, 7.9, -10.0)), ((8.0, 16.0, 8.0), (7.95, 0.0, 7.9)), ((8.0, 8.0, 8.0), (0.0, 0.0, 0.0))]


@pytest.mark.parametrize("storage,algo", [("hashtable", "longestaxis"), ("hashtable", "original"), ("vcs", "original")])
def test_render_from_region_corner_cameras(probe, storage, algo):
    """Cameras sitting exactly on a corner shared by eight regions (scale 8: (128, 64, 0), (64, 128, 64), (64, 64, 64)) looking
    along the faces: the frames where rays are rebased onto exactly 64.0.  The hash table is defined everywhere there (no cluster
    table to overrun, a key with a coordinate of 64 matches nothing) and so is the original algorithm; VCS + longest axis is left
    out because the reference's exists test is undefined at x = 64 (DESIGN.md 4)."""
    xyz, rgb = probe
    kind = oracle_kind()
    po.set_lighting(kind)
    ref, s = build_oracle(kind, xyz, rgb, storage), build_product(xyz, rgb, storage)
    s.set_statistics(True)
    for o, l in REGION_CORNER_CAMERAS:
        cam = api.Camera(o, l, (0.0, 1.0, 0.0), 60.0, np.float32(320) / np.float32(180))
        got = s.render(320, 180, algo, cam, scale=8, want_hits=True)
        st = s.get_statistics()
        want = ref.render(cam.data, 320, 180, algo, scale=8, want_counters=True)
        assert np.array_equal(got["hits"], want["hits"]), (storage, algo, o, int((got["hits"] != want["hits"]).any(-1).sum()))
        assert np.array_equal(got["rgb"], want["rgb"]), (storage, algo, o)
        assert (st["exist_checks"], st["exist_false"], st["lookups"]) == tuple(int(v) for v in want["counters"][:3]), (storage, algo, o)
    s.close()


def test_kernels_equal_their_host_compile_in_the_undefined_corner(probe):
    """VCS + longest axis from the region-corner cameras: the reference's exists test is undefined at x = 64 there, so no oracle can
    be matched -- but the kernels must still do exactly what their own source does when compiled for the host (tests/hostsim: same
    headers, same guard padding): deterministic, inside the allocations, and identical between the state machine and the host."""
    xyz, rgb = probe
    po.set_lighting("sim")
    sim, s = build_oracle("sim", xyz, rgb, "vcs"), build_product(xyz, rgb, "vcs")
    po._lib("sim").sim_set_flat(1)
    s.set_statistics(True)
    for o, l in REGION_CORNER_CAMERAS:
        cam = api.Camera(o, l, (0.0, 1.0, 0.0), 60.0, np.float32(320) / np.float32(180))
        got = s.render(320, 180, "longestaxis", cam, scale=8, want_hits=True)
        st = s.get_statistics()
        want = sim.render(cam.data, 320, 180, "longestaxis", scale=8, want_counters=True)
        assert np.array_equal(got["hits"], want["hits"]) and np.array_equal(got["rgb"], want["rgb"]), o
        assert (st["exist_checks"], st["exist_false"], st["lookups"]) == tuple(int(v) for v in want["counters"][:3]), o
    s.close()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("algo", ["original", "longestaxis"])
def test_trace_fuzz_from_grid_aligned_origins(algo):
    """Random rays from origins on cluster faces / integer coordinates (not on region-face corners, where the reference itself is
    undefined): many of them crawl (the oracle executes > 10^8 cluster-skip iterations here), a few cross a binade boundary while
    crawling -- the situations in which the first crawl_skip was off by one iteration.  Colours, hit voxels and event counters
    must equal the C oracle's."""
    po.set_lighting("orc")
    xyz, rgb = scenes.sparse_shells(256, 32, seed=9, fill_pct=45)
    s, ref = build_product(xyz, rgb, "vcs"), build_oracle("orc", xyz, rgb, "vcs")
    s.set_statistics(True)
    for i, origin in enumerate([(48.0, 240.0, 232.0), (208.0, 224.0, 16.0), (63.0, 39.0, 4.0)]):
        rays = scenes.random_rays(60000 if i == 0 else 30000, origin, seed=205 - i)   # ray 51980 of the first set crosses x = 32 while crawling
        got, want = s.trace_rays(rays, algo, want_hits=True), ref.trace_rays(rays, algo, want_counters=True)
        st = s.get_statistics()
        assert np.array_equal(got["colour"], want["colour"]) and np.array_equal(got["hits"], want["hits"]), origin
        assert (st["exist_checks"], st["exist_false"], st["lookups"]) == tuple(int(v) for v in want["counters"][:3]), origin
    s.close()
