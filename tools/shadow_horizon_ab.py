"""A/B of the shadow horizon map (vrm_core.cuh HorizonView) on the GPU, in one process: two handles of the bench scene, one created
with VRM_SHADOW_HORIZON=0 (every lit shadow ray walks out of the scene) and one with the map, render bench.py's view sequence in
alternating order for several rounds.  Each frame: L2 flushed (512 MiB write), then one CUDA event pair around the render.  Also the
structure build time (which includes the map) with and without it, on the bench terrain, the 2048^3 shells and the config 5 scene.

    python tools/shadow_horizon_ab.py [--rounds 5] [--views 20] [--out profiles/shadow_horizon_b200.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from voxelraymarcher_b200 import api  # noqa: E402
import bench  # noqa: E402


def handle(horizon):
    os.environ["VRM_SHADOW_HORIZON"] = "1" if horizon else "0"
    s = api.VoxelScene(0)
    del os.environ["VRM_SHADOW_HORIZON"]
    s.set_stream(torch.cuda.current_stream().cuda_stream)
    return s


def build_ms(fill, horizon, reps=3):
    out = []
    for _ in range(reps):
        s = handle(horizon)
        fill(s)
        s.synchronize()
        out.append(s.generate_voxel_scene("vcs"))
        s.close()
    return min(out)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--views", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    W, H = bench.WIDTH, bench.HEIGHT
    arms = {"off": handle(False), "on": handle(True)}
    for s in arms.values():
        s.generate_terrain(bench.SCENE_SIZE, bench.SCENE_SEED)
        s.generate_voxel_scene(bench.STORAGE)
    cams = [bench.orbit_camera(api, bench.view_of(k, 0, 1)) for k in range(a.views)]
    frame = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in cams]
    for s in arms.values():  # warm-up: every view once
        for c in cams:
            s.render_device(W, H, bench.ALGORITHM, c, frame.data_ptr())
    torch.cuda.synchronize()
    per = {"off": [], "on": []}
    for r in range(a.rounds):
        for name in (("off", "on") if r % 2 == 0 else ("on", "off")):
            s = arms[name]
            for c, (e0, e1) in zip(cams, ev):
                flush.fill_(r & 0xFF)
                e0.record(); s.render_device(W, H, bench.ALGORITHM, c, frame.data_ptr()); e1.record()
            torch.cuda.synchronize()
            per[name].append(float(np.mean([e0.elapsed_time(e1) for e0, e1 in ev])))
        print(f"round {r}: off {per['off'][-1]:.4f} ms/frame, on {per['on'][-1]:.4f} ms/frame", flush=True)
    off, on = np.array(per["off"]), np.array(per["on"])
    ratios = on / off
    res = {"card": card(), "workload": bench.workload_config()["workload"], "views": [bench.view_of(k, 0, 1) for k in range(a.views)],
           "method": "alternating handles per round, L2 flushed before every frame, one CUDA event pair per frame; ms = mean over the views",
           "ms_per_frame": {"off": per["off"], "on": per["on"]},
           "mean_ms": {"off": float(off.mean()), "on": float(on.mean())},
           "gain_pct": float(100.0 * (1.0 - on.mean() / off.mean())),
           "ratio_on_off": {"min": float(ratios.min()), "max": float(ratios.max())},
           "noise_pct_off_rounds": float(100.0 * (off.max() - off.min()) / off.mean())}
    for s in arms.values():
        s.close()
    del flush
    torch.cuda.synchronize()
    scenes = {"terrain512": lambda s: s.generate_terrain(bench.SCENE_SIZE, bench.SCENE_SEED),
              "shells2048": lambda s: s.generate_sparse_shells(2048, 64, 7, 35),
              "config5_shells1024": lambda s: s.generate_sparse_shells(1024, 64, 11, 35)}
    res["build_ms"] = {k: {"off": build_ms(f, False), "on": build_ms(f, True)} for k, f in scenes.items()}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
