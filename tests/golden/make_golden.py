"""Generates the committed golden fixtures.

    python tests/golden/make_golden.py            reference_golden.npz: the stand-in scenes at 160x90, rendered by the UNMODIFIED
                                                  reference built for the host (oracle/_ref/libvrm_ref_host.so, see oracle/ref_host.cpp;
                                                  needs a reference checkout, see oracle/Makefile)
    python tests/golden/make_golden.py configs    config_golden.npz: a seeded sample (tests/common.config_sample) of every frame and ray
                                                  buffer of tests/test_configs_gpu.py at full size -- hit records, RGB, and the four event
                                                  counters where that test compares them -- rendered by the strongest checker present (oracle_kind(); needs the built
                                                  library for the cameras, not a GPU)
The reference ships no golden vectors of its own (SURVEY.md F7); these pin the oracle and the CUDA path to the
reference's behaviour."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from tests.common import (COMBOS, GOLDEN_DIR, MINI_CAMERAS, PROBE_CAMERAS, build_oracle, camera, config_sample, lookup_queries,  # noqa: E402
                          oracle_kind, po, scenes)

W, H = 160, 90


def configs():
    from tests.test_configs_gpu import CONFIG4_VIEWS, config3_camera, config5_rays, orbit_camera_2048
    from voxelraymarcher_b200 import api
    kind = oracle_kind()
    out = {"checker": np.array(kind)}

    def frames(xyz, rgb, storages, algos, cams, scale, k=kind, counters=True):
        po.set_lighting(k)
        for storage in storages:
            ref = build_oracle(k, xyz, rgb, storage)
            for tag, cam, w, h in cams:
                for algo in algos:
                    r = ref.render(cam.data, w, h, algo, scale=scale, want_counters=True)
                    idx = config_sample(w * h)
                    key = f"{tag}_{storage}_{algo}"
                    out[f"{key}_hits"] = r["hits"].reshape(-1, 4)[idx]
                    out[f"{key}_rgb"] = r["rgb"].reshape(-1, 3)[idx]
                    if counters:
                        out[f"{key}_counters"] = r["counters"][:4].astype(np.int64)
                    print(key, flush=True)
            ref.close()

    xyz, rgb = scenes.probe_scene()
    frames(xyz, rgb, ["hashtable"], ["original"], [("config1", api.Camera.reference_default(1280, 720), 1280, 720)], 8)
    frames(xyz, rgb, ["hashtable", "vcs"], ["original", "longestaxis"], [("config2", api.Camera.reference_default(1920, 1080), 1920, 1080)], 8)
    xyz, rgb = scenes.terrain(512, 1234)
    frames(xyz, rgb, ["vcs", "hashtable"], ["longestaxis", "original"], [("config3", config3_camera(), 3840, 2160)], 1)
    xyz, rgb = scenes.sparse_shells(2048, 64, seed=7, fill_pct=35)
    frames(xyz, rgb, ["vcs"], ["longestaxis", "original"], [(f"config4_view{v}", orbit_camera_2048(v, 1920, 1080), 1920, 1080) for v in CONFIG4_VIEWS], 1,
           k="refgx" if po.available("refgx") else kind, counters=False)
    xyz, rgb = scenes.sparse_shells(1024, 64, seed=11, fill_pct=35)
    rays = config5_rays()
    idx = config_sample(rays.shape[0])
    po.set_lighting(kind)
    ref = build_oracle(kind, xyz, rgb, "vcs")
    for algo in ("longestaxis", "original"):
        r = ref.trace_rays(rays, algo, want_counters=True)
        out[f"config5_vcs_{algo}_hits"] = r["hits"][idx]
        out[f"config5_vcs_{algo}_colour"] = r["colour"][idx]
        out[f"config5_vcs_{algo}_counters"] = r["counters"][:4].astype(np.int64)
    ref.close()
    np.savez_compressed(os.path.join(GOLDEN_DIR, "config_golden.npz"), **out)
    print("wrote", os.path.join(GOLDEN_DIR, "config_golden.npz"), len(out), "arrays, checker", kind)


def main():
    assert po.available("refh"), "build oracle/_ref first (make -C oracle ref)"
    po.set_lighting("refh")
    out = {}
    for name, (xyz, rgb), scale in (("probe", scenes.probe_scene(), 8), ("mini", scenes.mini_scene(), 1)):
        q = lookup_queries(xyz, 4000, seed=7)
        out[f"{name}_queries"] = q
        for storage in ("hashtable", "vcs"):
            ref = build_oracle("refh", xyz, rgb, storage)
            info = ref.info()
            out[f"{name}_{storage}_info"] = np.array([info["diameter"], info["min_coord"], info["filled"]], np.int64)
            val, ex = ref.lookup(q)
            out[f"{name}_{storage}_lookup"] = val
            out[f"{name}_{storage}_exists"] = ex
            cams = PROBE_CAMERAS if name == "probe" else MINI_CAMERAS
            for ci, (o, l, fov) in enumerate(cams):
                cam = camera(o, l, fov, W, H, "refh")
                out[f"{name}_cam{ci}"] = cam
                for algo in ("original", "longestaxis"):
                    r = ref.render(cam, W, H, algo, scale=scale)
                    out[f"{name}_{storage}_{algo}_cam{ci}_rgb"] = r["rgb"]
                    out[f"{name}_{storage}_{algo}_cam{ci}_hits"] = r["hits"]
            ref.close()
    # lighting variants on the probe scene (point light on / shadows off), reference camera
    xyz, rgb = scenes.probe_scene()
    cam = camera(*PROBE_CAMERAS[1], W, H, "refh")
    for tag, kw in (("point", dict(use_point=True, position=(60.0, 90.0, 80.0))), ("noshadow", dict(use_shadows=False))):
        po.set_lighting("refh", **kw)
        for storage, algo in COMBOS:
            ref = build_oracle("refh", xyz, rgb, storage)
            r = ref.render(cam, W, H, algo, scale=8)
            out[f"probe_{storage}_{algo}_{tag}_rgb"] = r["rgb"]
            ref.close()
    po.set_lighting("refh")
    np.savez_compressed(os.path.join(GOLDEN_DIR, "reference_golden.npz"), **out)
    print("wrote", os.path.join(GOLDEN_DIR, "reference_golden.npz"), len(out), "arrays")


if __name__ == "__main__":
    if sys.argv[1:] == ["configs"]:
        configs()
    else:
        main()
