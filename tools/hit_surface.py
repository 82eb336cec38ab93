"""Cost of the hit-surface pass (vrm_hit_surface_views_device, csrc/vrm_surface.cu) next to the render that produces its input.

    python tools/hit_surface.py [--reps 30] [--out profiles/hit_surface_b200.json]

Two workloads, both on bench.py's scene (512^3 terrain, VCS + longest axis) and cameras: one 3840x2160 frame (orbit view 0, the camera
travels in the kernel arguments) and a 64-view 1920x1080 orbit batch (one launch, cameras uploaded).  Each is timed with CUDA events on
the scene's stream (5 warm-up calls, median of --reps): the render with its hit map, and the surface pass reading that hit map.  Bytes
are what the pass must move: 16 B of hit record read, 4 B of depth and 1 B of face written per pixel (rays are rebuilt from the camera).
The working sets (174 MB at 4K, 2.8 GB for the batch) exceed the 126 MB L2, so the pass streams from HBM; the share is of the B200 data
sheet's 7.7 TB/s.  Device name and power limit are read in the same run.
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
from voxelraymarcher_b200 import api  # noqa: E402

HBM_TBS = 7.7
BYTES_PER_PIXEL = 16 + 4 + 1


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (f.strip() for f in out.split(","))
        return dict(name=name, power_limit=power, sm_clock_max=clock)
    except Exception as e:  # noqa: BLE001
        return dict(name=None, power_limit=None, error=str(e))


def median_ms(torch, fn, reps, warmup=5):
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
    return float(np.median(times)), float(np.min(times)), float(np.max(times))


def workload(torch, s, name, cams, w, h, reps):
    n = len(cams)
    rgb = torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda")
    hits = torch.empty((n, h, w, 4), dtype=torch.int32, device="cuda")
    depth = torch.empty((n, h, w), dtype=torch.float32, device="cuda")
    face = torch.empty((n, h, w), dtype=torch.uint8, device="cuda")
    render = lambda: s.render_views_device(w, h, bench.ALGORITHM, cams, rgb.data_ptr(), hits.data_ptr())  # noqa: E731
    surface = lambda: s.hit_surface_views_device(hits.data_ptr(), cams, w, h, depth.data_ptr(), face.data_ptr())  # noqa: E731
    render_ms = median_ms(torch, render, reps)
    surface_ms = median_ms(torch, surface, reps)
    render()
    surface()
    torch.cuda.synchronize()
    px = n * w * h
    nbytes = px * BYTES_PER_PIXEL
    gbs = nbytes / (surface_ms[0] * 1e-3) / 1e9
    hit_share = float(hits[..., 3].float().mean().item())
    return dict(workload=name, views=n, width=w, height=h, pixels=px, hit_fraction=round(hit_share, 4),
                render_ms_median=round(render_ms[0], 4), render_ms_min=round(render_ms[1], 4), render_ms_max=round(render_ms[2], 4),
                surface_ms_median=round(surface_ms[0], 4), surface_ms_min=round(surface_ms[1], 4), surface_ms_max=round(surface_ms[2], 4),
                surface_over_render=round(surface_ms[0] / render_ms[0], 4), bytes=nbytes, surface_gbs=round(gbs, 1),
                share_of_hbm_peak=round(gbs / (HBM_TBS * 1e3), 4))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "hit_surface_b200.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    s = api.VoxelScene(0)
    s.set_stream(torch.cuda.current_stream().cuda_stream)
    s.generate_terrain(bench.SCENE_SIZE, bench.SCENE_SEED)
    s.generate_voxel_scene(bench.STORAGE)
    results = [workload(torch, s, "4k_single_view", [bench.orbit_camera(api, 0)], bench.WIDTH, bench.HEIGHT, a.reps)]
    orbit = [api.Camera(bench.orbit_camera(api, v).data[:3], bench.ORBIT_CENTRE, (0.0, 1.0, 0.0), 60.0, np.float32(1920) / np.float32(1080))
             for v in range(bench.ORBIT_VIEWS)]
    results.append(workload(torch, s, "orbit_64x1080p", orbit, 1920, 1080, a.reps))
    out = dict(tool="tools/hit_surface.py", device=device_info(), hbm_peak_tbs=HBM_TBS, bytes_per_pixel=BYTES_PER_PIXEL, reps=a.reps,
               scene=dict(size=bench.SCENE_SIZE, seed=bench.SCENE_SEED, storage=bench.STORAGE, algorithm=bench.ALGORITHM), results=results)
    s.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
