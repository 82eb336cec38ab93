"""GPU tier: every render and trace pipeline the library can select, against the oracle.

`launch_render_t` / `launch_trace_t` (csrc/vrm_render.cu) pick one pipeline per storage x algorithm combination, and the environment
switches read at `vrm_scene_create` (INTEGRATION.md 5) force any other.  The per-ray arithmetic of the nested, flat and lean forms is
covered by their host compile (tests/test_hostsim.py); what differs between the pipelines is the GPU orchestration around it -- the
persistent queue's refill, the lean kernels' park bitmap and resume, the three shadow-queue consumers and how they write a frame, the
defer queue, band launches and the splitting of view batches and ray lists into launches.  This file runs every selectable form
through those paths: bit-exact frames, hit maps and colours, and equal event counters, against the oracle or against the same output
computed another way (a device frame, single views, separate ray ranges, the stored full-size samples of tests/golden/config_golden.npz).

Every oracle output is computed once per module (`oracle` fixture) and shared by all the forms compared with it."""
import os

import numpy as np
import pytest

from tests.common import COMBOS, GOLDEN_DIR, PROBE_CAMERAS, build_oracle, config_sample, oracle_kind, po, scenes
from tests.test_configs_gpu import config3_camera, orbit_camera_2048
from tests.test_hostsim import axis_aligned_rays, crawl_scene_and_rays, pingpong_scene_and_rays
from voxelraymarcher_b200 import api

pytestmark = pytest.mark.gpu

# Every switch a form may set: cleared before each scene is created, so only the form's own values are in effect.
SWITCHES = ("VRM_RENDER_MODE", "VRM_SHADOW_FORM", "VRM_TRACE_SORT", "VRM_TRACE_FUSED", "VRM_PINNED_DMA", "VRM_WSTORE_REMOTE",
            "VRM_BULK_STORE", "VRM_DEFER_CAPACITY", "VRM_VIEW_BATCH_BYTES")

# Render pipelines (launch_render_t).  Under statistics mode 3 falls back to mode 2 (vrm_render.cu: the event counters live in the
# generic machine), so the counters of mode 3 cannot be checked: its colours and hits are checked without statistics.
RENDER_FORMS = [
    ("mode0-persistent", {"VRM_RENDER_MODE": "0"}),
    ("mode1-shadow0", {"VRM_RENDER_MODE": "1", "VRM_SHADOW_FORM": "0"}),
    ("mode1-shadow1", {"VRM_RENDER_MODE": "1", "VRM_SHADOW_FORM": "1"}),
    ("mode1-shadow2", {"VRM_RENDER_MODE": "1", "VRM_SHADOW_FORM": "2"}),
    ("mode2-fused", {"VRM_RENDER_MODE": "2"}),
    ("mode3-lean", {"VRM_RENDER_MODE": "3"}),
    ("mode4-shadow0", {"VRM_RENDER_MODE": "4", "VRM_SHADOW_FORM": "0"}),
    ("mode4-shadow1", {"VRM_RENDER_MODE": "4", "VRM_SHADOW_FORM": "1"}),
    ("mode4-shadow2", {"VRM_RENDER_MODE": "4", "VRM_SHADOW_FORM": "2"}),
]

# Trace pipelines (launch_trace_t).  The default sorts batches of >= 1024 rays and runs the fused kernel for VCS + longest axis;
# VRM_TRACE_FUSED=0 / VRM_TRACE_SORT=0 give the per-lane machine + refill shadow queue there.  Mode 3 as above.
TRACE_FORMS = [
    ("default", {}),
    ("unfused", {"VRM_TRACE_FUSED": "0"}),
    ("unsorted", {"VRM_TRACE_SORT": "0"}),
    ("mode1-shadow0", {"VRM_RENDER_MODE": "1", "VRM_SHADOW_FORM": "0"}),
    ("mode1-shadow1", {"VRM_RENDER_MODE": "1", "VRM_SHADOW_FORM": "1"}),
    ("mode1-shadow2", {"VRM_RENDER_MODE": "1", "VRM_SHADOW_FORM": "2"}),
    ("mode2-shadow0", {"VRM_RENDER_MODE": "2", "VRM_SHADOW_FORM": "0"}),
    ("mode2-shadow1", {"VRM_RENDER_MODE": "2", "VRM_SHADOW_FORM": "1"}),
    ("mode3-lean", {"VRM_RENDER_MODE": "3"}),
]

# The trace forms that run the defer queue for VCS + longest axis (mode 2, fused or not)
DEFER_TRACE_FORMS = [f for f in TRACE_FORMS if f[0] in ("default", "unfused", "unsorted", "mode2-shadow0", "mode2-shadow1")]

render_forms = pytest.mark.parametrize("form,env", RENDER_FORMS, ids=[f for f, _ in RENDER_FORMS])
trace_forms = pytest.mark.parametrize("form,env", TRACE_FORMS, ids=[f for f, _ in TRACE_FORMS])
combos = pytest.mark.parametrize("storage,algo", COMBOS, ids=[f"{s}-{a}" for s, a in COMBOS])

COUNTER_KEYS = ("exist_checks", "exist_false", "lookups", "lookup_hits")

# lighting variants: (product setup_constant_values kwargs, oracle set_lighting kwargs)
LIGHTING = {
    "sun": ({}, {}),
    "point": (dict(use_point_light=True, light_position=(60.0, 90.0, 80.0)), dict(use_point=True, position=(60.0, 90.0, 80.0))),
    "noshadow": (dict(use_shadows=False), dict(use_shadows=False)),
}


def counted(form):
    return not form.startswith("mode3")


def counters(st, k=4):
    return [st[key] for key in COUNTER_KEYS[:k]]


def form_scene(monkeypatch, env, xyz, rgb, storage):
    """A scene built with exactly the switches in env (they are read at vrm_scene_create)."""
    for name in SWITCHES:
        monkeypatch.delenv(name, raising=False)
    for name, value in env.items():
        monkeypatch.setenv(name, value)
    s = api.VoxelScene(0)
    s.add_voxels(xyz, rgb)
    s.generate_voxel_scene(storage)
    return s


def probe_camera(ci, w, h):
    o, l, fov = PROBE_CAMERAS[ci]
    return api.Camera(o, l, (0.0, 1.0, 0.0), fov, np.float32(w) / np.float32(h))


def shells_rays():
    return scenes.random_rays(200000, (130.0, 97.0, 121.0), seed=42)


def pingpong_padded():
    """The ping-pong rays followed by ordinary rays: >= 1024 rays, so that the default VCS + longest-axis trace sorts them and runs
    the fused kernel (smaller batches take the caller's order and the per-lane machine)."""
    xyz, rgb, rays = pingpong_scene_and_rays()
    pad = scenes.random_rays(1100, (40.0, 70.0, 40.0), seed=19)
    return xyz, rgb, np.concatenate([rays, pad]).astype(np.float32)


SCENES = {
    "probe": lambda: scenes.probe_scene() + (axis_aligned_rays(),),
    "shells": lambda: scenes.sparse_shells(256, 64, seed=7, fill_pct=50) + (shells_rays(),),
    "crawl": crawl_scene_and_rays,
    "pingpong": pingpong_padded,
}


class Oracle:
    """The oracle's outputs, each computed once: keyed by (scene, storage, algorithm, camera or ray set, size, lighting, translation)."""

    def __init__(self):
        self.kind = oracle_kind()
        self.data, self.built, self.out = {}, {}, {}

    def scene(self, name):
        if name not in self.data:
            self.data[name] = SCENES[name]()
        return self.data[name]

    def _ref(self, name, storage):
        if (name, storage) not in self.built:
            xyz, rgb, _ = self.scene(name)
            self.built[(name, storage)] = build_oracle(self.kind, xyz, rgb, storage)
        return self.built[(name, storage)]

    def render(self, storage, algo, ci, w, h, light="sun", translation=(0.0, 0.0, 0.0)):
        key = ("render", "probe", storage, algo, ci, w, h, light, translation)
        if key not in self.out:
            po.set_lighting(self.kind, **LIGHTING[light][1])
            cam = probe_camera(ci, w, h)
            self.out[key] = self._ref("probe", storage).render(cam.data, w, h, algo, scale=8, translation=translation, want_counters=True)
        return self.out[key]

    def trace(self, name, storage, algo, rays_tag, rays, scale=1, threads=None):
        key = ("trace", name, storage, algo, rays_tag, scale)
        if key not in self.out:
            po.set_lighting(self.kind)
            self.out[key] = self._ref(name, storage).trace_rays(rays, algo, scale=scale, want_counters=True, threads=threads)
        return self.out[key]

    def close(self):
        for r in self.built.values():
            r.close()


@pytest.fixture(scope="module")
def oracle():
    o = Oracle()
    yield o
    o.close()


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(GOLDEN_DIR, "config_golden.npz"))


# ---- 1. render matrix on the probe scene -------------------------------------------------------------------------------------------------


@combos
@render_forms
def test_render_forms_match_oracle(monkeypatch, oracle, form, env, storage, algo):
    """Every render form x combination on the probe scene (scale 8): the four probe cameras at an aligned and a ragged size, a point light,
    no shadows, a non-zero translation and sizes below one tile.  Hit maps and RGB bit-exact without and with statistics; the
    reference-comparable counters equal the oracle's; the as-executed counters give the same frame with no more work."""
    xyz, rgb, _ = oracle.scene("probe")
    s = form_scene(monkeypatch, env, xyz, rgb, storage)
    cases = [(ci, w, h, "sun", (0.0, 0.0, 0.0)) for (w, h) in ((640, 360), (333, 187)) for ci in range(len(PROBE_CAMERAS))]
    cases += [(1, 320, 180, "point", (0.0, 0.0, 0.0)), (1, 320, 180, "noshadow", (0.0, 0.0, 0.0)), (1, 320, 180, "sun", (3.5, -2.25, 7.0))]
    cases += [(0, w, h, "sun", (0.0, 0.0, 0.0)) for (w, h) in ((33, 5), (7, 3), (1, 1))]
    for ci, w, h, light, tr in cases:
        tag = (form, storage, algo, ci, w, h, light, tr)
        want = oracle.render(storage, algo, ci, w, h, light, tr)
        s.setup_constant_values(**LIGHTING[light][0])
        cam = probe_camera(ci, w, h)
        s.set_statistics(False)
        got = s.render(w, h, algo, cam, scale=8, translation=tr, want_hits=True)
        assert np.array_equal(got["hits"], want["hits"]), (tag, int((got["hits"] != want["hits"]).any(-1).sum()))
        assert np.array_equal(got["rgb"], want["rgb"]), tag
        if not counted(form):
            continue
        s.set_statistics(True)
        got = s.render(w, h, algo, cam, scale=8, translation=tr, want_hits=True)
        st = s.get_statistics()
        assert np.array_equal(got["hits"], want["hits"]) and np.array_equal(got["rgb"], want["rgb"]), tag
        assert counters(st) == [int(v) for v in want["counters"][:4]], tag
        assert st["rays"] == w * h
        if light == "sun" and (w, h) == (640, 360):
            s.set_statistics(True, as_executed=True)
            ex = s.render(w, h, algo, cam, scale=8, translation=tr)
            st2 = s.get_statistics()
            assert np.array_equal(ex["rgb"], want["rgb"]), tag
            assert st2["rays"] == st["rays"] and st2["lookup_hits"] <= st["lookup_hits"] and st2["exist_checks"] <= st["exist_checks"], tag
            if ci == 1:
                assert 0 < st2["exist_checks"] < st["exist_checks"], tag
    s.close()


# ---- 2. frame placement at 4K -----------------------------------------------------------------------------------------------------------

PLACEMENTS = [  # (name, extra switches, page-locked frame)
    ("pageable", {}, False),                           # the handle's page-locked staging frame, three 6 MB bands at 4K
    ("pinned", {}, True),                              # stores into the mapped frame (CTA-staged rows, or a local frame + copy)
    ("dma1", {"VRM_PINNED_DMA": "1"}, True),           # device frame + copy-engine bands
    ("dma3", {"VRM_PINNED_DMA": "3"}, True),
    ("dma8", {"VRM_PINNED_DMA": "8"}, True),
    ("wstore", {"VRM_WSTORE_REMOTE": "1"}, True),      # per-warp stores into the mapped frame
    ("nobulk", {"VRM_BULK_STORE": "0"}, True),         # staged rows as ordinary stores
]


@pytest.fixture(scope="module")
def pinned4k():
    import torch
    return torch.zeros((2160, 3840, 3), dtype=torch.uint8).pin_memory()


@combos
@render_forms
def test_frame_placements_equal_the_device_frame(monkeypatch, oracle, pinned4k, form, env, storage, algo):
    """A 3840x2160 frame of the probe scene rendered into pageable memory (three bands), into page-locked memory, through 1, 3 and 8
    copy-engine bands, with per-warp remote stores and without bulk copies equals the device-frame render of the same form, hits
    included; the counters of the banded calls equal those of the single device-frame launch."""
    import torch
    xyz, rgb, _ = oracle.scene("probe")
    w, h = 3840, 2160
    cam = probe_camera(1, w, h)
    s = form_scene(monkeypatch, env, xyz, rgb, storage)
    dev = torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda:0")
    dev_hits = torch.zeros((h, w, 4), dtype=torch.int32, device="cuda:0")
    s.render_device(w, h, algo, cam, dev.data_ptr(), dev_hits.data_ptr(), scale=8)
    s.synchronize()
    want_rgb, want_hits = dev.cpu().numpy(), dev_hits.cpu().numpy()
    assert want_hits[..., 3].sum() > 100_000
    want_st = None
    if counted(form):
        s.set_statistics(True)
        s.render_device(w, h, algo, cam, dev.data_ptr(), scale=8)
        want_st = counters(s.get_statistics()) + [w * h]
        s.set_statistics(False)
    pinned = pinned4k.numpy()
    for name, extra, page_locked in PLACEMENTS:
        t = form_scene(monkeypatch, {**env, **extra}, xyz, rgb, storage) if extra else s
        for stats in ((False, True) if counted(form) else (False,)):
            t.set_statistics(stats)
            out = pinned if page_locked else np.empty((h, w, 3), np.uint8)
            out.fill(7)
            got = t.render(w, h, algo, cam, scale=8, want_hits=not stats, rgb_out=out)
            assert np.array_equal(out, want_rgb), (form, name, stats, int((out != want_rgb).any(-1).sum()))
            if stats:
                st = t.get_statistics()
                assert counters(st) + [st["rays"]] == want_st, (form, name)
            else:
                assert np.array_equal(got["hits"], want_hits), (form, name)
        if t is not s:
            t.close()
    s.close()


# ---- 3. view batches across a launch boundary -------------------------------------------------------------------------------------------


@combos
@render_forms
def test_view_batch_across_a_launch_boundary(monkeypatch, oracle, form, env, storage, algo):
    """Six 3840x2160 views in one call run as two launches (4 + 2 views: the shadow-ray queue holds 2^25 records).  The batch, and the
    same batch into every second slot of a 12-slot buffer, equal the single-view renders, hit maps included; the batch's counters are
    the sum of the single views' counters."""
    import torch
    xyz, rgb, _ = oracle.scene("probe")
    w, h, n = 3840, 2160, 6
    cams = [api.Camera((14.0 - 2.5 * v, 9.0 - 0.5 * v, 12.0 - 3.0 * v), (4.0, 3.0, 2.0), (0.0, 1.0, 0.0), 60.0, np.float32(w) / np.float32(h))
            for v in range(n)]
    s = form_scene(monkeypatch, env, xyz, rgb, storage)
    one = torch.zeros((n, h, w, 3), dtype=torch.uint8, device="cuda:0")
    one_hits = torch.zeros((n, h, w, 4), dtype=torch.int32, device="cuda:0")
    batch = torch.full((n, h, w, 3), 7, dtype=torch.uint8, device="cuda:0")
    batch_hits = torch.full((n, h, w, 4), 7, dtype=torch.int32, device="cuda:0")
    strided = torch.full((2 * n, h, w, 3), 7, dtype=torch.uint8, device="cuda:0")
    strided_hits = torch.full((2 * n, h, w, 4), 7, dtype=torch.int32, device="cuda:0")
    for stats in ((False, True) if counted(form) else (False,)):
        s.set_statistics(stats)
        total = [0, 0, 0, 0, 0]
        for v in range(n):
            s.render_device(w, h, algo, cams[v], one[v].data_ptr(), one_hits[v].data_ptr(), scale=8)
            if stats:
                st = s.get_statistics()
                total = [a + b for a, b in zip(total, counters(st) + [st["rays"]])]
        s.render_views_device(w, h, algo, cams, batch.data_ptr(), batch_hits.data_ptr(), scale=8)
        if stats:
            st = s.get_statistics()
            assert counters(st) + [st["rays"]] == total, form
        s.render_views_device(w, h, algo, cams, strided.data_ptr(), strided_hits.data_ptr(), scale=8, view_stride=2)
        s.synchronize()
        assert (one_hits[..., 3] != 0).sum(dim=(1, 2)).min().item() > 100_000
        for v in range(n):
            assert torch.equal(batch[v], one[v]) and torch.equal(batch_hits[v], one_hits[v]), (form, stats, v)
            assert torch.equal(strided[2 * v], one[v]) and torch.equal(strided_hits[2 * v], one_hits[v]), (form, stats, v)
        assert (strided[1::2] == 7).all() and (strided_hits[1::2] == 7).all()
    s.close()


# ---- 4. trace matrix --------------------------------------------------------------------------------------------------------------------


def check_trace(s, want, rays, algo, form, ncounters, scale=1, tag=None):
    s.set_statistics(False)
    got = s.trace_rays(rays, algo, scale=scale, want_hits=True)
    bad = int((got["hits"] != want["hits"]).any(-1).sum())
    assert bad == 0, (tag, form, algo, f"{bad} hit records differ")
    assert np.array_equal(got["colour"], want["colour"]), (tag, form, algo)
    if counted(form) and ncounters:
        s.set_statistics(True)
        got = s.trace_rays(rays, algo, scale=scale, want_hits=True)
        st = s.get_statistics()
        assert np.array_equal(got["hits"], want["hits"]) and np.array_equal(got["colour"], want["colour"]), (tag, form, algo)
        assert counters(st, ncounters) == [int(v) for v in want["counters"][:ncounters]], (tag, form, algo)
        assert st["rays"] == rays.shape[0]
    return got


@combos
@trace_forms
def test_trace_forms_match_oracle_sparse_shells(monkeypatch, oracle, form, env, storage, algo):
    """200 000 incoherent rays in the 256^3 sparse-shell scene (config 5 at oracle-friendly size): colours, hit records and counters."""
    xyz, rgb, rays = oracle.scene("shells")
    want = oracle.trace("shells", storage, algo, "random", rays)
    assert want["hits"][:, 3].sum() > 1000
    s = form_scene(monkeypatch, env, xyz, rgb, storage)
    check_trace(s, want, rays, algo, form, 4, tag="shells")
    s.close()


@combos
@trace_forms
def test_trace_forms_axis_aligned_rays(monkeypatch, oracle, form, env, storage, algo):
    """Rays with exactly-zero direction components (inf / NaN in the reference's divisions) terminate in every form and equal the
    reference's host build."""
    xyz, rgb, rays = oracle.scene("probe")
    want = oracle.trace("probe", storage, algo, "axis-aligned", rays, threads=1)
    s = form_scene(monkeypatch, env, xyz, rgb, storage)
    check_trace(s, want, rays, algo, form, 0, tag="axis-aligned")
    s.close()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("algo", ["original", "longestaxis"])
@trace_forms
def test_trace_forms_crawl_fast_forward(monkeypatch, oracle, form, env, algo):
    """Rays stuck on the face of an empty VCS cluster (~5e7 reference iterations): every form fast-forwards or crawls to the same
    colours, hit voxels and counters."""
    xyz, rgb, rays = oracle.scene("crawl")
    want = oracle.trace("crawl", "vcs", algo, "crawl", rays)
    s = form_scene(monkeypatch, env, xyz, rgb, "vcs")
    check_trace(s, want, rays, algo, form, 4, tag="crawl")
    s.close()


@pytest.mark.timeout(600)
@trace_forms
def test_trace_forms_region_face_pingpong(monkeypatch, oracle, form, env):
    """Rays that hop across a region face twice per cycle (VCS + longest axis).  The state machines park them in the defer queue and
    fast-forward them; the nested form (mode 1) has no ping-pong probe and crawls like the reference -- exact, only slower."""
    xyz, rgb, rays = oracle.scene("pingpong")
    want = oracle.trace("pingpong", "vcs", "longestaxis", "pingpong", rays)
    s = form_scene(monkeypatch, env, xyz, rgb, "vcs")
    check_trace(s, want, rays, "longestaxis", form, 3, tag="pingpong")
    s.close()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("form,env", DEFER_TRACE_FORMS, ids=[f for f, _ in DEFER_TRACE_FORMS])
def test_trace_forms_full_defer_queue(monkeypatch, oracle, form, env):
    """The ping-pong case with a defer queue of 3 records for every trace form that parks rays: the rays that find it full crawl on
    in their kernel, with the same results and counters."""
    xyz, rgb, rays = oracle.scene("pingpong")
    want = oracle.trace("pingpong", "vcs", "longestaxis", "pingpong", rays)
    s = form_scene(monkeypatch, {**env, "VRM_DEFER_CAPACITY": "3"}, xyz, rgb, "vcs")
    check_trace(s, want, rays, "longestaxis", form, 3, tag="pingpong, 3 defer slots")
    s.close()


# ---- 5. the ray-chunk boundary ----------------------------------------------------------------------------------------------------------

CHUNK = 1 << 25          # rays per trace launch (vrm_launch_trace)
N_CHUNKED = CHUNK + 4099


@pytest.fixture(scope="module")
def chunk_rays():
    """N_CHUNKED rays (world units, the probe scene at scale 8) generated on the device, so the host holds no 800 MB copy."""
    import torch
    g = torch.Generator(device="cuda:0")
    g.manual_seed(2025)
    o = torch.rand((N_CHUNKED, 3), generator=g, device="cuda:0") * torch.tensor([24.0, 14.0, 24.0], device="cuda:0") - torch.tensor([4.0, 2.0, 6.0], device="cuda:0")
    d = torch.randn((N_CHUNKED, 3), generator=g, device="cuda:0")
    d = d / d.norm(dim=1, keepdim=True)
    return torch.cat([o, d], 1).contiguous()


@pytest.mark.timeout(900)
@combos
@pytest.mark.parametrize("order", ["sorted", "unsorted"])
def test_trace_across_the_ray_chunk_boundary(monkeypatch, oracle, chunk_rays, order, storage, algo):
    """2^25 + 4099 rays run as two launches.  Colours and hits equal those of two separate traces of [0, 2^25) and [2^25, n); the whole
    call's counters are the sum of the parts'; the 20 000 rays around index 2^25 equal the oracle's."""
    import torch
    xyz, rgb, _ = oracle.scene("probe")
    s = form_scene(monkeypatch, {} if order == "sorted" else {"VRM_TRACE_SORT": "0"}, xyz, rgb, storage)

    def trace(first, n, stats):
        s.set_statistics(stats)
        colour = torch.zeros(n, dtype=torch.int32, device="cuda:0")
        hits = torch.zeros((n, 4), dtype=torch.int32, device="cuda:0")
        s.trace_rays_device(chunk_rays[first:].data_ptr(), n, algo, colour.data_ptr(), hits.data_ptr(), scale=8)
        s.synchronize()
        st = s.get_statistics() if stats else None
        return colour, hits, (counters(st) + [st["rays"]] if stats else None)

    for stats in (False, True):
        whole = trace(0, N_CHUNKED, stats)
        a = trace(0, CHUNK, stats)
        b = trace(CHUNK, N_CHUNKED - CHUNK, stats)
        assert torch.equal(whole[0][:CHUNK], a[0]) and torch.equal(whole[0][CHUNK:], b[0]), (order, stats)
        assert torch.equal(whole[1][:CHUNK], a[1]) and torch.equal(whole[1][CHUNK:], b[1]), (order, stats)
        assert (whole[1][CHUNK:, 3] != 0).sum().item() > 10 and (whole[1][:CHUNK, 3] != 0).sum().item() > 100_000
        if stats:
            assert whole[2] == [x + y for x, y in zip(a[2], b[2])], order
        lo, hi = CHUNK - 10000, CHUNK + 10000
        rays = chunk_rays[lo:hi].cpu().numpy()
        want = oracle.trace("probe", storage, algo, "chunk-boundary", rays, scale=8)
        assert np.array_equal(whole[1][lo:hi].cpu().numpy(), want["hits"]), (order, stats)
        assert np.array_equal(whole[0][lo:hi].cpu().numpy().view(np.uint32), want["colour"]), (order, stats)
        del whole, a, b
    s.close()


# ---- 6. full size -----------------------------------------------------------------------------------------------------------------------


def _sample(t, n):
    """The rows of a device tensor at the stored sample positions of an output of n positions (tests.common.config_sample)."""
    import torch
    idx = torch.from_numpy(config_sample(n)).to(t.device)
    return t.reshape(n, -1)[idx].cpu().numpy()


def _render_dev(s, w, h, algo, cam):
    import torch
    rgb = torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda:0")
    hits = torch.zeros((h, w, 4), dtype=torch.int32, device="cuda:0")
    s.render_device(w, h, algo, cam, rgb.data_ptr(), hits.data_ptr())
    s.synchronize()
    return rgb, hits


@pytest.mark.timeout(900)
@pytest.mark.parametrize("storage", ["vcs", "hashtable"])
def test_full_size_terrain_every_render_form(monkeypatch, golden, storage):
    """The 512^3 terrain (generate_terrain(512, 1234); this comparison is what pins the GPU generator to scenes.terrain at 512) at
    3840x2160 with config 3's camera: every render form and both algorithms give the default form's frame and hit map, the stored
    samples of config3_{storage}_{algo} and its stored counters."""
    import torch
    w, h = 3840, 2160
    cam = config3_camera()
    frames = {}
    for form, env in [("default", {})] + RENDER_FORMS:
        for name in SWITCHES:
            monkeypatch.delenv(name, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        s = api.VoxelScene(0)
        s.generate_terrain(512, 1234)
        s.generate_voxel_scene(storage)
        for algo in ("longestaxis", "original"):
            key = f"config3_{storage}_{algo}"
            rgb, hits = _render_dev(s, w, h, algo, cam)
            assert np.array_equal(_sample(hits, w * h), golden[f"{key}_hits"]), (form, algo)
            assert np.array_equal(_sample(rgb, w * h), golden[f"{key}_rgb"]), (form, algo)
            if form == "default":
                frames[algo] = (rgb, hits)
            else:
                assert torch.equal(rgb, frames[algo][0]), (form, algo, int((rgb != frames[algo][0]).any(-1).sum()))
                assert torch.equal(hits, frames[algo][1]), (form, algo, int((hits != frames[algo][1]).any(-1).sum()))
            if counted(form):
                s.set_statistics(True)
                rgb2, _ = _render_dev(s, w, h, algo, cam)
                st = s.get_statistics()
                s.set_statistics(False)
                assert torch.equal(rgb2, frames[algo][0]), (form, algo)
                assert counters(st) == golden[f"{key}_counters"].tolist(), (form, algo)
        s.close()


@pytest.mark.timeout(1500)
def test_full_size_orbit_view_every_render_form(monkeypatch, golden):
    """View 3 of the 2048^3 orbit (config 4, VCS, 1920x1080), the one full-size scene where the defer queue parks rays: every render form
    and both algorithms give the default form's frame and the stored samples of config4_view3_vcs_{algo}."""
    import torch
    w, h = 1920, 1080
    cam = orbit_camera_2048(3, w, h)
    frames = {}
    for form, env in [("default", {})] + RENDER_FORMS:
        for name in SWITCHES:
            monkeypatch.delenv(name, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        s = api.VoxelScene(0)
        s.generate_sparse_shells(2048, 64, 7, 35)
        s.generate_voxel_scene("vcs")
        for algo in ("longestaxis", "original"):
            key = f"config4_view3_vcs_{algo}"
            rgb, hits = _render_dev(s, w, h, algo, cam)
            assert np.array_equal(_sample(hits, w * h), golden[f"{key}_hits"]), (form, algo)
            assert np.array_equal(_sample(rgb, w * h), golden[f"{key}_rgb"]), (form, algo)
            if form == "default":
                frames[algo] = (rgb, hits)
            else:
                assert torch.equal(rgb, frames[algo][0]) and torch.equal(hits, frames[algo][1]), (form, algo)
        s.close()


def test_traced_build_gives_the_same_scene(monkeypatch, oracle):
    """VRM_BUILD_TRACE=1 (stage marks on stderr, a synchronisation per stage) builds the same scene."""
    xyz, rgb, _ = oracle.scene("probe")
    for storage in ("vcs", "hashtable"):
        plain = form_scene(monkeypatch, {}, xyz, rgb, storage)
        monkeypatch.setenv("VRM_BUILD_TRACE", "1")
        traced = form_scene(monkeypatch, {}, xyz, rgb, storage)
        monkeypatch.delenv("VRM_BUILD_TRACE")
        assert traced.info() == plain.info()
        q = np.concatenate([xyz, xyz + 1, xyz - 7]).astype(np.int32)
        assert np.array_equal(traced.lookup(q)[0], plain.lookup(q)[0])
        cam = probe_camera(1, 320, 180)
        a, b = traced.render(320, 180, "longestaxis", cam, scale=8, want_hits=True), plain.render(320, 180, "longestaxis", cam, scale=8, want_hits=True)
        assert np.array_equal(a["rgb"], b["rgb"]) and np.array_equal(a["hits"], b["hits"])
        plain.close(); traced.close()
