"""Voxel lists out of a built scene (vrm_scene_read_voxels_device), timed against what a user does without it (DESIGN.md 3.5).

Cases, both storage types: the whole 512^3 terrain (BASELINE.json config 3, 27-bit sort keys), the whole 2048^3 sparse-shell scene
(config 4, 33-bit keys: the 64-bit sort) and a 512^3 box inside it.  Baseline on the same box: vrm_scene_read_box_device into a dense
uint32 volume, then torch ``nonzero`` and a gather of the colours.  A dense box of more than 2^30 cells (the whole 2048^3 box: 34 GB)
is read in x-slabs of 2^30 cells, one slab buffer reused, and the slab times are summed.  Both outputs are compared on the device.

Device work is timed with CUDA events on a dedicated stream after warm-up (medians); read_voxels_device includes its one host round
trip (the count).  The split between count, fill, sort and write comes from a separate torch.profiler run (kernel times, grouped by
launch order: everything before the fill kernel is the count, between fill and write the sort).  Bytes model (per case, computed here
from the listed voxels):
  region-table entries of the touched cells (4 B)
  VCS: per listed region its 64-byte cluster mask; per touched occupied cluster its 128-byte header line, read by the count AND the fill
       pass; 4 B colour per voxel (fill)
  hash table: per listed region its 16-byte descriptor and all its slots, 8 B x 2 x (c + c/4 + 2) for c voxels, read by both passes
  unit counts: 4 B written + scanned (3 x 4 B) per unit, 64 units per listed region
  fill: key + colour written per voxel; sort: per pass (3 K + 8) B per voxel (histogram reads the key, scatter reads and writes key +
  colour; K = key bytes); write: key + colour read, 16 B written per voxel.

    python tools/voxels_out.py [--out profiles/voxels_out_b200.json] [--reps 10]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench import measured_peak  # noqa: E402
from dense_io import Timer, gpu_identity, stats  # noqa: E402
from voxelraymarcher_b200 import api  # noqa: E402

EMPTY = api.EMPTY
SLAB_CELLS = 1 << 30


def make_scene(name, storage, stream):
    s = api.VoxelScene(0)
    s.set_stream(stream.cuda_stream)
    if name == "terrain512":
        s.generate_terrain(512, 1234)
    else:
        s.generate_sparse_shells(2048, 64, 7, 35)
    s.generate_voxel_scene(storage)
    s.synchronize()
    return s


def bits_for(e):
    b = 0
    while (1 << b) < e:
        b += 1
    return b


def bytes_model(s, storage, origin, dims, xyz, all_region_counts):
    info = s.info()
    n = len(xyz)
    t0, t1 = 64 * info["min_coord"], 64 * (info["min_coord"] + info["diameter"])
    lo = [max(o, t0) for o in origin]
    hi = [min(o + d, t1) for o, d in zip(origin, dims)]
    touched_cells = int(np.prod([((h - 1) >> 6) - (lo_ >> 6) + 1 for lo_, h in zip(lo, hi)]))
    regions = unique_rows(xyz >> 6)
    # regions listed = non-null regions the box touches; the voxel list only shows those holding a voxel IN the box (a lower bound)
    listed = len(regions)
    key_bits = sum(bits_for(h - lo_) for lo_, h in zip(lo, hi))
    K = 4 if key_bits <= 32 else 8
    passes = (key_bits + 8) // 9
    parts = dict(region_table=4 * touched_cells, unit_counts=16 * 64 * listed)
    if storage == "vcs":
        clusters = len(unique_rows(xyz >> 3))
        parts.update(cluster_masks=64 * listed, header_lines=2 * 128 * clusters, colours=4 * n)
    else:
        c = np.array([all_region_counts[tuple(r)] for r in regions.tolist()], np.int64)
        parts.update(hash_descriptors=16 * listed, hash_slots=2 * int((8 * 2 * (c + c // 4 + 2)).sum()))
    parts.update(fill_writes=(K + 4) * n, sort=passes * (3 * K + 8) * n, write_reads=(K + 4) * n, output=16 * n)
    return dict(key_bits=key_bits, key_bytes=K, sort_passes=passes, touched_region_cells=touched_cells, listed_regions_lower_bound=listed,
                parts=parts, total=int(sum(parts.values())))


def unique_rows(a, return_counts=False):
    """np.unique(a, axis=0) of an (n, 3) integer array through one packed int64 key (much faster for tens of millions of rows)."""
    a = np.asarray(a, np.int64)
    if len(a) == 0:
        return (np.zeros((0, 3), np.int64), np.zeros(0, np.int64)) if return_counts else np.zeros((0, 3), np.int64)
    lo = a.min(0)
    span = a.max(0) - lo + 1
    key = ((a[:, 0] - lo[0]) * span[1] + (a[:, 1] - lo[1])) * span[2] + (a[:, 2] - lo[2])
    u, c = np.unique(key, return_counts=True)
    rows = np.stack([u // (span[1] * span[2]) + lo[0], (u // span[2]) % span[1] + lo[1], u % span[2] + lo[2]], 1)
    return (rows, c) if return_counts else rows


def region_counts(xyz):
    r, c = unique_rows(xyz >> 6, return_counts=True)
    return {tuple(k): int(v) for k, v in zip(r.tolist(), c.tolist())}


def phase_split(s, origin, dims, d_xyz, d_rgb, cap):
    """Kernel times of one call by phase, from torch.profiler (kernel launch order)."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        s.read_voxels_device(origin, dims, d_xyz.data_ptr(), d_rgb.data_ptr(), cap)
        s.synchronize()
        torch.cuda.synchronize()
    ks = sorted([(e.time_range.start, e.time_range.elapsed_us(), e.name) for e in prof.events() if e.device_type == DeviceType.CUDA
                 and "emcpy" not in e.name and "emset" not in e.name])
    phase, out, names = "count", {"count": 0.0, "fill": 0.0, "sort": 0.0, "write": 0.0}, {}
    for _, us, name in ks:
        if "voxels_units_kernel" in name and ("Lb1E" in name or "true" in name):
            phase = "fill"
        elif phase == "fill" and "voxels_units_kernel" not in name:
            phase = "sort"
        if "voxels_write_kernel" in name:
            phase = "write"
        out[phase] += us / 1e3
        names.setdefault(phase, set()).add(name.replace("(anonymous namespace)::", "").split("(")[0][:90])
    return dict(kernel_ms=out, kernels={k: sorted(v) for k, v in names.items()})


def baseline(s, origin, dims, stream, tm):
    """read_box_device + nonzero + gather, in x-slabs of at most 2^30 cells; returns (ms, xyz, rgb) of the device results."""
    import torch
    plane = dims[1] * dims[2]
    slab = max(1, min(dims[0], SLAB_CELLS // plane))
    buf = torch.empty((slab, dims[1], dims[2]), dtype=torch.int32, device="cuda")
    xs, cs = [], []
    ms = 0.0
    for x0 in range(0, dims[0], slab):
        nx = min(slab, dims[0] - x0)
        v = buf[:nx]
        e0 = tm.event()
        s.read_box_device((origin[0] + x0, origin[1], origin[2]), (nx, dims[1], dims[2]), v.data_ptr())
        mask = v != EMPTY
        idx = mask.nonzero()
        rgb = v[mask]
        xyz = (idx + torch.tensor([origin[0] + x0, origin[1], origin[2]], device="cuda")).to(torch.int32)
        e1 = tm.event()
        stream.synchronize()
        ms += e0.elapsed_time(e1)
        xs.append(xyz)
        cs.append(rgb)
        del mask, idx
    return ms, torch.cat(xs), torch.cat(cs), dict(slabs=(dims[0] + slab - 1) // slab, slab_cells=slab * plane)


def run_case(name, origin, dims, stream, reps, peak):
    import torch
    tm = Timer(stream)
    rows = []
    for storage in ("vcs", "hashtable"):
        s = make_scene(name, storage, stream)
        with torch.cuda.stream(stream):
            if origin is None:
                origin, dims = s.scene_box()
            n = s.count_voxels(origin, dims)
            d_xyz = torch.empty((n, 3), dtype=torch.int32, device="cuda")
            d_rgb = torch.empty((n,), dtype=torch.int32, device="cuda")
            for _ in range(3):
                s.read_voxels_device(origin, dims, d_xyz.data_ptr(), d_rgb.data_ptr(), n)
            ms = []
            for _ in range(reps):
                e0 = tm.event()
                s.read_voxels_device(origin, dims, d_xyz.data_ptr(), d_rgb.data_ptr(), n)
                e1 = tm.event()
                stream.synchronize()
                ms.append(e0.elapsed_time(e1))
            cnt = []
            for _ in range(reps):
                e0 = tm.event()
                s.count_voxels(origin, dims)
                e1 = tm.event()
                stream.synchronize()
                cnt.append(e0.elapsed_time(e1))
            base_ms, bx, brgb, slabs = baseline(s, origin, dims, stream, tm)  # warm-up
            bms = []
            for _ in range(max(2, reps // 3)):
                del bx, brgb
                t, bx, brgb, slabs = baseline(s, origin, dims, stream, tm)
                bms.append(t)
            same = bool(torch.equal(bx, d_xyz) and torch.equal(brgb, d_rgb))
            del bx, brgb
            try:
                split = phase_split(s, origin, dims, d_xyz, d_rgb, n)
            except Exception as e:  # noqa: BLE001
                split = dict(error=repr(e))
            xyz = d_xyz.cpu().numpy()
        whole = xyz if tuple(dims) == tuple(s.scene_box()[1]) else s.read_voxels()[0]   # per-region voxel counts of the hash model
        model = bytes_model(s, storage, origin, dims, xyz, region_counts(whole))
        med = stats(ms)["median_ms"]
        gbs = model["total"] / (med * 1e-3) / 1e9
        row = dict(scene=name, storage=storage, origin=list(origin), dims=list(dims), voxels=n, unique_voxels=s.info()["unique_voxels"],
                   read_voxels_device=stats(ms), count_only=stats(cnt), baseline_read_box_nonzero=dict(**stats(bms), **slabs),
                   speedup_vs_baseline=stats(bms)["median_ms"] / med, outputs_equal_baseline=same, phases=split,
                   bytes_model=model, roofline=dict(bound="hbm", achieved_gbs=gbs, peak_gbs=peak, frac=gbs / peak))
        print(json.dumps(row), flush=True)
        rows.append(row)
        s.close()
        del d_xyz, d_rgb, xyz, whole
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the whole result to this JSON file")
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available() or not api.device_available():
        raise SystemExit("voxels_out.py needs a CUDA device")
    peak, peak_src = measured_peak()
    ident = gpu_identity()
    print(json.dumps(ident), flush=True)
    stream = torch.cuda.Stream()
    cases = []
    cases += run_case("terrain512", None, None, stream, a.reps, peak)
    cases += run_case("sparse_shells2048", None, None, stream, a.reps, peak)
    cases += run_case("sparse_shells2048", (768, 768, 768), (512, 512, 512), stream, a.reps, peak)
    result = dict(gpu=ident, hbm_peak_gbs=peak, hbm_peak_source=peak_src, reps=a.reps, cases=cases)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        json.dump(result, open(a.out, "w"), indent=1)
        print("wrote", a.out)


if __name__ == "__main__":
    main()
