"""Development aid: which blocks of the state machine does a WARP of the headline render kernel execute per pass?  Lockstep simulation of
march_scene_flat_warp on the CPU (tests/hostsim: the product's own traversal source compiled for the host) over sampled 8x4 tiles of the
bench frame (512^3 terrain, 3840x2160, view 0), VCS + longest axis.

    python tools/warp_profile.py [--size 512] [--stride 4] [--view 0]
    python tools/warp_profile.py --views 20 --horizon both   # passes per tile over bench.py's view sequence, shadow horizon map off / on

The library is tests/horizon_sim.py's host build (tests/hostsim plus the horizon map's entry points); terrain cameras are made there with
Camera.cuh's formula, as api.Camera, so the tool needs no GPU library.
"""
import argparse
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from voxelraymarcher_b200 import scenes  # noqa: E402
from tests import horizon_sim  # noqa: E402
import bench  # noqa: E402

CATS = ["region", "head", "test", "jump", "next", "cluster", "nullreg", "hitwait", "done"]


def camera(lib, view):
    org, at, up, fov, aspect = bench._orbit_args(view)
    out = np.zeros(15, np.float32)
    f3 = [np.ascontiguousarray(v, np.float32) for v in (org, at, up)]
    lib.hz_camera_make(*(v.ctypes.data_as(ctypes.c_void_p) for v in f3), ctypes.c_float(fov), ctypes.c_float(aspect), out.ctypes.data_as(ctypes.c_void_p))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--stride", type=int, default=4)
    ap.add_argument("--view", type=int, default=0)
    ap.add_argument("--threads", type=int, default=os.cpu_count())
    ap.add_argument("--regroup", default="", help="budget:maxLanes[,budget:maxLanes...]: simulate abandon + re-trace of long-tailed tiles (sim_regroup_profile)")
    ap.add_argument("--compact", default="", help="tiles per CTA, e.g. 2,4,8: simulate packing the shadow rays of a CTA's tiles into full warps (sim_cta_compact_profile)")
    ap.add_argument("--scene", default="terrain", choices=["terrain", "shells2048"], help="shells2048: BASELINE configs[3], one 1080p view of its orbit")
    ap.add_argument("--horizon", default="off", choices=["off", "on", "both"], help="--views: shadow rays end at the horizon map (vrm_core.cuh HorizonView)")
    ap.add_argument("--views", type=int, default=0, help="terrain: passes per tile over the first N views of bench.py's sequence (bench.view_of) instead of one profile")
    a = ap.parse_args()
    lib = horizon_sim.load()
    if a.scene == "terrain":
        xyz, rgb = scenes.terrain(a.size, bench.SCENE_SEED)
    else:
        xyz, rgb = scenes.sparse_shells(2048, 64, seed=7, fill_pct=35)
    h = ctypes.c_void_p(lib.sim_scene_create())
    xyz = np.ascontiguousarray(xyz, np.int32); rgb = np.ascontiguousarray(rgb, np.uint32)
    lib.sim_scene_add_voxels(h, xyz.ctypes.data_as(ctypes.c_void_p), rgb.ctypes.data_as(ctypes.c_void_p), ctypes.c_uint64(len(rgb)))
    assert lib.sim_scene_build_vcs_fast(h) == 0
    light = [np.array(v, np.float32) for v in ((0.57735026, 0.57735026, 0.57735026), (1, 1, 1), (10, 10, -10))]
    d = np.zeros(3, np.float32)
    lib.sim_make_unit_vector(np.array([1.0, 1.0, 1.0], np.float32).ctypes.data_as(ctypes.c_void_p), d.ctypes.data_as(ctypes.c_void_p))
    W, H = bench.WIDTH, bench.HEIGHT
    if a.scene == "terrain":
        camv = camera(lib, a.view)
    else:
        from voxelraymarcher_b200 import api
        W, H = 1920, 1080
        camv = np.ascontiguousarray(bench.orbit_views_2048(api, W, H)[a.view].data, np.float32)
    tr = np.zeros(3, np.float32)
    if a.views:
        views = [bench.view_of(k, 0, 1) for k in range(a.views)]
        modes = [0, 1] if a.horizon == "both" else [int(a.horizon == "on")]
        per = {}
        for m in modes:
            for v in views:
                cv = camera(lib, v)
                tot = np.zeros(3, np.uint64)
                assert lib.hz_warp_passes(h, cv.ctypes.data_as(ctypes.c_void_p), tr.ctypes.data_as(ctypes.c_void_p), 1, W, H, a.stride, m,
                                          tot.ctypes.data_as(ctypes.c_void_p), a.threads) == 0
                per[(m, v)] = (int(tot[1]) / int(tot[0]), int(tot[2]) / int(tot[0]))
                print(f"horizon {'on ' if m else 'off'} view {v:2d}: passes/tile {per[(m, v)][0]:6.2f} (shadow {per[(m, v)][1]:6.2f})", flush=True)
        for m in modes:
            p = np.mean([per[(m, v)][0] for v in views]); sp = np.mean([per[(m, v)][1] for v in views])
            print(f"horizon {'on ' if m else 'off'}: mean over {len(views)} views: passes/tile {p:.3f}, shadow passes/tile {sp:.3f}")
        if len(modes) == 2:
            off = np.mean([per[(0, v)][0] for v in views]); on = np.mean([per[(1, v)][0] for v in views])
            print(f"passes per tile: {100 * (off - on) / off:.1f} % fewer with the horizon map")
        return
    if a.compact:
        for tpc in (int(v) for v in a.compact.split(",")):
            out = np.zeros(7, np.uint64)
            rc = lib.sim_cta_compact_profile(h, camv.ctypes.data_as(ctypes.c_void_p), tr.ctypes.data_as(ctypes.c_void_p), 1, W, H, a.stride, tpc,
                                             out.ctypes.data_as(ctypes.c_void_p), a.threads)
            assert rc == 0
            ctas, pp, sp, spk, slp, srays, worst = (int(v) for v in out)
            tiles = ctas * tpc
            print(f"tiles/CTA {tpc}: primary passes/tile {pp / tiles:.2f}, shadow passes/tile {sp / tiles:.2f} (lanes/pass {slp / max(sp, 1):.1f}) -> packed {spk / tiles:.2f}; "
                  f"all passes {100 * (pp + spk) / (pp + sp):.1f} %; shadow rays/tile {srays / tiles:.2f}; worst tile of a CTA / mean primary passes {worst * tpc / pp:.2f}")
        return
    if a.regroup:
        for spec in a.regroup.split(","):
            budget, lanes_max = (int(v) for v in spec.split(":"))
            out = np.zeros(6, np.uint64)
            rc = lib.sim_regroup_profile(h, camv.ctypes.data_as(ctypes.c_void_p), tr.ctypes.data_as(ctypes.c_void_p), 1, W, H, a.stride, budget, lanes_max,
                                         out.ctypes.data_as(ctypes.c_void_p), a.threads)
            assert rc == 0
            tiles, p1, p0, listed, p2, lp2 = (int(v) for v in out)
            print(f"budget {budget:4d} lanes<= {lanes_max:2d}: passes/tile {p0 / tiles:7.2f} -> phase 1 {p1 / tiles:7.2f} + phase 2 {p2 / tiles:6.2f} = {(p1 + p2) / tiles:7.2f} "
                  f"({100 * (p1 + p2) / p0:5.1f} %), re-traced pixels {100 * listed / (tiles * 32):5.1f} %, phase-2 lanes/pass {lp2 / max(p2, 1):5.1f}")
        return
    hist = np.zeros(512, np.uint64); lanes = np.zeros((512, 9), np.uint64); tot = np.zeros(4, np.uint64)
    rc = lib.sim_warp_profile(h, camv.ctypes.data_as(ctypes.c_void_p), tr.ctypes.data_as(ctypes.c_void_p), 1, W, H, a.stride,
                              hist.ctypes.data_as(ctypes.c_void_p), lanes.ctypes.data_as(ctypes.c_void_p), tot.ctypes.data_as(ctypes.c_void_p), a.threads)
    assert rc == 0
    tiles, passes, shade, lanepasses = (int(v) for v in tot)
    print(f"tiles {tiles}  passes/tile {passes / tiles:.2f}  shading passes/tile {shade / tiles:.2f}  marching lanes/pass {lanepasses / passes:.2f}")
    print("passes in which a category is present, lanes in it when present:")
    for k, name in enumerate(CATS[:8]):
        p = sum(int(hist[s]) for s in range(512) if (s >> k) & 1)
        l = sum(int(lanes[s, k]) for s in range(512))
        print(f"  {name:9s} {100 * p / passes:6.2f} % of passes, {l / max(p, 1):5.1f} lanes")
    shadow = sum(int(hist[s]) for s in range(512) if s & 256)
    print(f"shadow-ray passes {100 * shadow / passes:.1f} % of passes")
    print("most frequent signatures (marching categories only; S = shadow-ray pass):")
    agg = {}
    for s in range(512):
        if hist[s]:
            m = s & 0x17F
            e = agg.setdefault(m, [0, np.zeros(9)])
            e[0] += int(hist[s]); e[1] += lanes[s].astype(np.float64)
    for m, (n, l) in sorted(agg.items(), key=lambda kv: -kv[1][0])[:25]:
        names = ("S " if m & 256 else "P ") + "+".join(CATS[k] for k in range(7) if (m >> k) & 1)
        print(f"  {100 * n / passes:6.2f} %  {names:40s} " + " ".join(f"{CATS[k][:4]}={l[k] / n:.1f}" for k in range(9) if l[k]))


if __name__ == "__main__":
    main()
