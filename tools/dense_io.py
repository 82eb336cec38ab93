"""Dense volumes in and out of a scene, timed against what a user does without them (DESIGN.md 3.4).

* Compaction: vrm_scene_add_dense_device + build of the 512^3 terrain as a dense uint32 volume on the GPU, against torch
  ``nonzero`` + vrm_scene_add_voxels_device + build and against ``nonzero`` + a host voxel list + vrm_scene_add_voxels + build.
* Box read: vrm_scene_read_box_device of a 512^3 box against vrm_lookup of every cell of it (a 12-byte host query per cell, the
  only way to read a scene back before), on the terrain ([0, 512)^3) and on a 512^3 box of the 2048^3 sparse_shells scene
  (BASELINE.json config 4), both storage types.

Device work is timed with CUDA events on a dedicated stream after warm-up; the host-buffer paths (vrm_lookup, vrm_scene_add_voxels)
with a host clock around work that ends in a synchronisation.  Achieved GB/s are over the bytes model below; the share is against
the HBM peak bench.py uses (MEASURED_PEAKS.json).  Bytes model:
  compaction: 8 B per cell (two streaming reads of the volume) + 16 B per voxel (xyz + colour written);
  box read:   4 B per cell written + VCS: one 128-byte header line per occupied cluster + 4 B per voxel (colour);
              hash table: one 16-byte probe pair per cell of an occupied cluster (the cluster filter passes it).

    python tools/dense_io.py [--out profiles/dense_io_b200.json] [--reps 10]

The result is printed as JSON lines; --out also writes it as one JSON file.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import measured_peak  # noqa: E402
from voxelraymarcher_b200 import api, scenes  # noqa: E402

EMPTY = api.EMPTY


def gpu_identity():
    import torch
    row = dict(device=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [f.strip() for f in q.split(",")]
        row.update(nvidia_smi_name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # noqa: BLE001
        row.update(power_limit=f"unavailable ({e})")
    return row


class Timer:
    """CUDA events on one stream."""

    def __init__(self, stream):
        import torch
        self.stream, self.torch = stream, torch

    def event(self):
        e = self.torch.cuda.Event(enable_timing=True)
        e.record(self.stream)
        return e


def terrain_volume_device(size=512, seed=1234):
    """scenes.terrain(size, seed) as a dense int32 (bit pattern uint32) volume on the GPU: vol[x, y, z] = colour(y) iff y < h[x, z]."""
    import torch
    h = torch.from_numpy(np.clip(scenes.terrain_heights(size, seed), 1, size - 1).astype(np.int32)).cuda()
    y = np.arange(size, dtype=np.int32)
    colour = torch.from_numpy(scenes._height_colour(y).astype(np.uint32).view(np.int32)).cuda()
    ys = torch.arange(size, dtype=torch.int32, device="cuda")
    return torch.where(ys[None, :, None] < h[:, None, :], colour[None, :, None], torch.tensor(EMPTY, dtype=torch.int32, device="cuda")).contiguous()


def stats(ms):
    ms = sorted(ms)
    return dict(median_ms=ms[len(ms) // 2], min_ms=ms[0], max_ms=ms[-1], n=len(ms))


def compaction(stream, reps, peak):
    import torch
    tm = Timer(stream)
    vol = terrain_volume_device()
    torch.cuda.synchronize()   # made on the default stream, used on `stream`
    dims = tuple(vol.shape)
    cells = vol.numel()
    out = {}
    with torch.cuda.stream(stream):
        voxels = int((vol != EMPTY).sum().item())
        model = 8 * cells + 16 * voxels
        for storage in ("vcs", "hashtable"):
            rows = {"add_dense_device": [], "nonzero_add_voxels_device": [], "nonzero_host_add_voxels": []}
            infos = {}
            for rep in range(reps + 2):
                # (1) the new path
                s = api.VoxelScene(0)
                s.set_stream(stream.cuda_stream)
                e0 = tm.event()
                n = s.add_dense_device(vol.data_ptr(), dims)
                e1 = tm.event()
                s.generate_voxel_scene(storage)
                e2 = tm.event()
                stream.synchronize()
                assert n == voxels
                infos["dense"] = s.info()
                s.close()
                t_dense = (e0.elapsed_time(e1), e1.elapsed_time(e2))
                # (2) torch nonzero -> device voxel list -> add_voxels_device
                s = api.VoxelScene(0)
                s.set_stream(stream.cuda_stream)
                e0 = tm.event()
                mask = vol != EMPTY
                xyz = mask.nonzero().to(torch.int32).contiguous()
                rgb = vol[mask].contiguous()
                s.add_voxels_device(xyz.data_ptr(), rgb.data_ptr(), xyz.shape[0])
                e1 = tm.event()
                s.generate_voxel_scene(storage)
                e2 = tm.event()
                stream.synchronize()
                infos["list_device"] = s.info()
                s.close()
                del mask, xyz, rgb
                t_dev = (e0.elapsed_time(e1), e1.elapsed_time(e2))
                # (3) torch nonzero -> host voxel list -> add_voxels (host clock: the list goes through host memory)
                s = api.VoxelScene(0)
                s.set_stream(stream.cuda_stream)
                stream.synchronize()
                t0 = time.perf_counter()
                mask = vol != EMPTY
                xyz = mask.nonzero().to(torch.int32).cpu().numpy()
                rgb = vol[mask].cpu().numpy().view(np.uint32)
                s.add_voxels(xyz, rgb)
                s.synchronize()
                t1 = time.perf_counter()
                s.generate_voxel_scene(storage)
                s.synchronize()
                t2 = time.perf_counter()
                infos["list_host"] = s.info()
                s.close()
                del mask, xyz, rgb
                t_host = ((t1 - t0) * 1e3, (t2 - t1) * 1e3)
                if rep >= 2:
                    rows["add_dense_device"].append(t_dense)
                    rows["nonzero_add_voxels_device"].append(t_dev)
                    rows["nonzero_host_add_voxels"].append(t_host)
            assert infos["dense"] == infos["list_device"] == infos["list_host"], infos
            res = {}
            for k, v in rows.items():
                res[k] = dict(add=stats([a for a, _ in v]), build=stats([b for _, b in v]), total=stats([a + b for a, b in v]),
                              clock="host perf_counter around synchronised work" if k == "nonzero_host_add_voxels" else "CUDA events")
            add_ms = res["add_dense_device"]["add"]["median_ms"]
            gbs = model / (add_ms * 1e-3) / 1e9
            res["add_dense_device"]["roofline"] = dict(bound="hbm", model_bytes=model, achieved_gbs=gbs, peak_gbs=peak, frac=gbs / peak,
                                                       note="add time includes the one host round trip that learns the count")
            res["speedup_add_vs_nonzero_device"] = res["nonzero_add_voxels_device"]["add"]["median_ms"] / add_ms
            res["speedup_add_vs_nonzero_host"] = res["nonzero_host_add_voxels"]["add"]["median_ms"] / add_ms
            res["speedup_total_vs_nonzero_host"] = res["nonzero_host_add_voxels"]["total"]["median_ms"] / res["add_dense_device"]["total"]["median_ms"]
            out[storage] = res
            print(json.dumps({"compaction": storage, **res}), flush=True)
    return dict(volume="terrain 512^3 (seed 1234) as a dense uint32 volume on the GPU", cells=cells, voxels=voxels, model_bytes=model, by_storage=out)


def box_cells(origin, dims):
    g = np.meshgrid(*[np.arange(o, o + d, dtype=np.int32) for o, d in zip(origin, dims)], indexing="ij")
    return np.ascontiguousarray(np.stack([a.ravel() for a in g], 1))


def box_read(stream, reps, peak):
    import torch
    tm = Timer(stream)
    cases = [("terrain512", (0, 0, 0)), ("sparse_shells2048", (768, 768, 768))]
    dims = (512, 512, 512)
    cells = int(np.prod(dims))
    out = []
    for name, origin in cases:
        coords = box_cells(origin, dims)
        for storage in ("vcs", "hashtable"):
            s = api.VoxelScene(0)
            s.set_stream(stream.cuda_stream)
            if name == "terrain512":
                s.generate_terrain(512, 1234)
            else:
                s.generate_sparse_shells(2048, 64, 7, 35)
            s.generate_voxel_scene(storage)
            with torch.cuda.stream(stream):
                d_out = torch.empty(dims, dtype=torch.int32, device="cuda")
                for _ in range(3):
                    s.read_box_device(origin, dims, d_out.data_ptr())
                ms = []
                for _ in range(reps):
                    e0 = tm.event()
                    s.read_box_device(origin, dims, d_out.data_ptr())
                    e1 = tm.event()
                    stream.synchronize()
                    ms.append(e0.elapsed_time(e1))
                box = d_out.cpu().numpy().view(np.uint32)
            occ = (box != EMPTY)
            voxels = int(occ.sum())
            clusters = int(occ.reshape(64, 8, 64, 8, 64, 8).any(axis=(1, 3, 5)).sum())
            if storage == "vcs":
                model = 4 * cells + 128 * clusters + 4 * voxels
                model_text = "4 B/cell written + 128 B/occupied cluster + 4 B/voxel"
            else:
                model = 4 * cells + 16 * 512 * clusters
                model_text = "4 B/cell written + 16 B probe pair per cell of an occupied cluster"
            # vrm_lookup of every cell: 12-byte host queries in, colour + exists out (host clock)
            s.lookup(coords[:1024])
            lk = []
            for _ in range(2):
                t0 = time.perf_counter()
                val, _ex = s.lookup(coords)
                lk.append((time.perf_counter() - t0) * 1e3)
            assert np.array_equal(val.reshape(dims), box), (name, storage, "read_box differs from lookup")
            med = stats(ms)["median_ms"]
            gbs = model / (med * 1e-3) / 1e9
            row = dict(scene=name, storage=storage, origin=origin, dims=dims, cells=cells, voxels=voxels, occupied_clusters=clusters,
                       read_box_device=stats(ms), lookup_every_cell_host=stats(lk), speedup_vs_lookup=stats(lk)["median_ms"] / med,
                       roofline=dict(bound="hbm", model=model_text, model_bytes=model, achieved_gbs=gbs, peak_gbs=peak, frac=gbs / peak,
                                     write_only_frac=(4 * cells) / (med * 1e-3) / 1e9 / peak))
            print(json.dumps(row), flush=True)
            out.append(row)
            s.close()
            del d_out, box, occ
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the whole result to this JSON file")
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available() or not api.device_available():
        raise SystemExit("dense_io.py needs a CUDA device")
    peak, peak_src = measured_peak()
    ident = gpu_identity()
    print(json.dumps(ident), flush=True)
    stream = torch.cuda.Stream()
    result = dict(gpu=ident, hbm_peak_gbs=peak, hbm_peak_source=peak_src, reps=a.reps,
                  compaction=compaction(stream, max(3, a.reps // 2), peak), box_read=box_read(stream, a.reps, peak))
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        json.dump(result, open(a.out, "w"), indent=1)
        print("wrote", a.out)


if __name__ == "__main__":
    main()
