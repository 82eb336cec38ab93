"""Throughput of the exact ray cast (vrm_cast_*_device, csrc/vrm_cast.cu) next to the reference walks plus hit surfaces on the same rays.

    python tools/cast_rays.py [--reps 20] [--out profiles/cast_rays_b200.json]

Workloads:
  * config 5: 3840x2160 scenes.random_rays from (543.5)^3 in the 1024^3 sparse shells (seed 11), VCS and hash table: cast_rays_device over
    [0, +inf) and over [0, 64] (early exit), against trace_rays_device (both algorithms) + hit_surface_rays_device on the same buffer;
  * bench.py's view 0 of the 512^3 terrain at 3840x2160: cast_views_device against render_device + hit_surface_views_device;
  * the 64-view 1920x1080 orbit of bench.py in one launch: cast_views_device against render_views_device + hit_surface_views_device.
Each call is timed with CUDA events on the scene's stream after 3 warm-up calls; the median of --reps is reported with min and max.  L2 is
not flushed between calls: the scene structures stay L2-resident as they do in a real stream of work, while the outputs (> 126 MB per call)
pass through HBM.  Device name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from voxelraymarcher_b200 import api, scenes  # noqa: E402


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (f.strip() for f in out.split(","))
        return dict(name=name, power_limit=power, sm_clock_max=clock)
    except Exception as e:  # noqa: BLE001
        return dict(name=None, power_limit=None, error=str(e))


def timed(torch, fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return dict(ms_median=round(float(np.median(times)), 4), ms_min=round(float(np.min(times)), 4), ms_max=round(float(np.max(times)), 4))


def rate(entry, n):
    entry["mrays_per_s"] = round(n / (entry["ms_median"] * 1e-3) / 1e6, 1)
    return entry


def config5(torch, storage, reps):
    s = api.VoxelScene(0)
    s.set_stream(torch.cuda.current_stream().cuda_stream)
    s.generate_sparse_shells(1024, 64, 11, 35)
    s.generate_voxel_scene(storage)
    rays = torch.from_numpy(scenes.random_rays(3840 * 2160, (512.0 + 31.5,) * 3, seed=42)).cuda()
    n = rays.shape[0]
    ranges64 = torch.tensor([0.0, 64.0], dtype=torch.float32, device="cuda").repeat(n, 1).contiguous()
    hits = torch.empty((n, 4), dtype=torch.int32, device="cuda")
    depth = torch.empty(n, dtype=torch.float32, device="cuda")
    face = torch.empty(n, dtype=torch.uint8, device="cuda")
    colour = torch.empty(n, dtype=torch.int32, device="cuda")
    out = (hits.data_ptr(), depth.data_ptr(), face.data_ptr(), colour.data_ptr())
    res = dict(workload=f"config5_{storage}", rays=n)
    res["cast"] = rate(timed(torch, lambda: s.cast_rays_device(rays.data_ptr(), n, None, *out), reps), n)
    res["cast_hit_fraction"] = round(float(hits[:, 3].float().mean().item()), 4)
    res["cast_t_far_64"] = rate(timed(torch, lambda: s.cast_rays_device(rays.data_ptr(), n, ranges64.data_ptr(), *out), reps), n)
    res["cast_t_far_64_hit_fraction"] = round(float(hits[:, 3].float().mean().item()), 4)
    surf = lambda: s.hit_surface_rays_device(hits.data_ptr(), rays.data_ptr(), n, depth.data_ptr(), face.data_ptr())  # noqa: E731
    for algo in ("longestaxis", "original"):
        tr = timed(torch, lambda: s.trace_rays_device(rays.data_ptr(), n, algo, colour.data_ptr(), hits.data_ptr()), reps)
        sf = timed(torch, surf, reps)
        tot = rate(dict(ms_median=round(tr["ms_median"] + sf["ms_median"], 4)), n)
        res[f"trace_{algo}"] = rate(tr, n)
        res[f"trace_{algo}_plus_surface"] = tot
    res["surface_pass"] = timed(torch, surf, reps)
    s.close()
    return res


def views(torch, s, name, cams, w, h, reps):
    nv = len(cams)
    n = nv * w * h
    rgb = torch.empty((nv, h, w, 3), dtype=torch.uint8, device="cuda")
    hits = torch.empty((nv, h, w, 4), dtype=torch.int32, device="cuda")
    depth = torch.empty((nv, h, w), dtype=torch.float32, device="cuda")
    face = torch.empty((nv, h, w), dtype=torch.uint8, device="cuda")
    colour = torch.empty((nv, h, w), dtype=torch.int32, device="cuda")
    out = (hits.data_ptr(), depth.data_ptr(), face.data_ptr(), colour.data_ptr())
    if nv == 1:
        render = lambda: s.render_device(w, h, bench.ALGORITHM, cams[0], rgb.data_ptr(), hits.data_ptr())  # noqa: E731
    else:
        render = lambda: s.render_views_device(w, h, bench.ALGORITHM, cams, rgb.data_ptr(), hits.data_ptr())  # noqa: E731
    surf = lambda: s.hit_surface_views_device(hits.data_ptr(), cams, w, h, depth.data_ptr(), face.data_ptr())  # noqa: E731
    res = dict(workload=name, views=nv, width=w, height=h, rays=n)
    res["cast"] = rate(timed(torch, lambda: s.cast_views_device(cams, w, h, *out), reps), n)
    res["cast_hit_fraction"] = round(float(hits[..., 3].float().mean().item()), 4)
    r = timed(torch, render, reps)
    sf = timed(torch, surf, reps)
    res["render"] = rate(r, n)
    res["surface_pass"] = sf
    res["render_plus_surface"] = rate(dict(ms_median=round(r["ms_median"] + sf["ms_median"], 4)), n)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cast_rays_b200.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    results = [config5(torch, st, a.reps) for st in ("vcs", "hashtable")]
    s = api.VoxelScene(0)
    s.set_stream(torch.cuda.current_stream().cuda_stream)
    s.generate_terrain(bench.SCENE_SIZE, bench.SCENE_SEED)
    s.generate_voxel_scene(bench.STORAGE)
    results.append(views(torch, s, "terrain512_view0_4k", [bench.orbit_camera(api, 0)], bench.WIDTH, bench.HEIGHT, a.reps))
    orbit = [api.Camera(bench.orbit_camera(api, v).data[:3], bench.ORBIT_CENTRE, (0.0, 1.0, 0.0), 60.0, np.float32(1920) / np.float32(1080))
             for v in range(bench.ORBIT_VIEWS)]
    results.append(views(torch, s, "terrain512_orbit_64x1080p", orbit, 1920, 1080, a.reps))
    s.close()
    out = dict(tool="tools/cast_rays.py", device=device_info(), l2_flushed=False, reps=a.reps, warmup=3,
               timing="CUDA events on the scene's stream, median of reps; '_plus_surface' entries add the two medians", results=results)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
