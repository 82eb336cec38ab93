#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json: primary Mrays/s and ms/frame at 4K on the 512^3
scene at 1/2/4/8 B200).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank per GPU)
    python bench.py --impl reference ...                      (the reference's own CPU implementation on the host cores)
    python bench.py ... --dump-outputs DIR                    (+ a seeded sample of the last timed step's frames, DIR/*.npy)

A step = one pass of the hot path over one batch of synthetic input = ONE 3840x2160 frame per GPU of the procedural
512^3 terrain (~32 M voxels, BASELINE.json configs[2]) with the reference CLI's default combination (Voxel Cluster Store +
longest-axis traversal, Main.cu:45-68), shadows on.  Frame (step k, rank r) is view (25 k + r * 64 / N) mod 64 of a 64-view
orbit whose view 0 is SURVEY.md 8d-3's camera: every rank renders DIFFERENT frames (VERDICT r01: sharding must not be measured on
replicated identical work), and the stride of 25 walks the orbit in a low-discrepancy order so that any K consecutive frames
sample it evenly and every rank's mean frame cost is the single GPU's.  The named single view itself is timed separately
(`single_view`).  The structure is built once per GPU, on the GPU, before the timed region and is replicated on every rank.

N > 1: the path's only exchange step -- finished frames arriving on rank 0 -- is fused into the render kernels (stores into rank
0's buffer over NVLink peer memory) and completion is a release store of a sequence number behind every frame, no collective:
ranks do not wait for each other between steps; rank 0's last step ends when every rank's last frame has landed.

value  = W*H*N*K / t, t = max over ranks of the summed per-step CUDA-event time; inputs and outputs resident in HBM.  L2 is
         flushed between steps (outside the per-step event pairs).
e2e    = the same metric through the host-buffer C-ABI call vrm_render (camera host -> device in the kernel arguments + frame D2H inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WIDTH, HEIGHT = 3840, 2160
SCENE_SIZE, SCENE_SEED = 512, 1234
STORAGE, ALGORITHM = "vcs", "longestaxis"       # the reference CLI's defaults (SURVEY.md F1)
ORBIT_CENTRE = (256.0, 64.0, 256.0)
ORBIT_RADIUS, ORBIT_HEIGHT, ORBIT_VIEWS = 498.0, 352.0, 64
METRIC = "primary_mrays_per_s_4k_512cube"
UNIT = "Mrays/s"


VIEW_STRIDE = 25     # odd: a permutation of the 64 views in a low-discrepancy order


def view_of(step: int, rank: int, world: int) -> int:
    """Every rank walks the SAME low-discrepancy sequence of orbit views (stride 25), rotated by rank * 64 / N: at any step the N ranks
    render N different views spaced evenly around the orbit, and every rank's K frames sample the orbit exactly as the single GPU's do
    (the first form, ((step * N + rank) * 25) mod 64, gave a rank only 64 / gcd(64, 25 N) = 8 distinct views at N = 8, whose mean cost
    differed by +-3 % between ranks: a sampling artefact in a max-over-ranks time)."""
    return (step * VIEW_STRIDE + rank * (ORBIT_VIEWS // max(1, world))) % ORBIT_VIEWS


def bind_to_gpu_numa_node(index: int):
    """Pin this rank's host threads to the CPUs next to its GPU (NVML affinity) BEFORE any page-locked buffer is allocated, so that
    the frames the kernels store over PCIe land in local host memory (N = 8: eight GPUs writing 25 MB frames at once)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [w * 64 + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:  # noqa: BLE001
        pass
    return None


def orbit_camera(api, view: int):
    """View `view` of a 64-view orbit around the terrain; view 0 is SURVEY.md §8d-3's camera (-96,352,-96)."""
    ang = np.float64(-0.75 * np.pi) + 2.0 * np.pi * (view % ORBIT_VIEWS) / ORBIT_VIEWS
    org = (float(np.float32(ORBIT_CENTRE[0] + ORBIT_RADIUS * np.cos(ang))), ORBIT_HEIGHT, float(np.float32(ORBIT_CENTRE[2] + ORBIT_RADIUS * np.sin(ang))))
    return api.Camera(org, ORBIT_CENTRE, (0.0, 1.0, 0.0), 60.0, np.float32(WIDTH) / np.float32(HEIGHT))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=float(max(mx)) if mx else None, reasons=sorted(reasons), samples=len(sm))


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def algorithmic_bytes(stats, storage):
    """SURVEY.md §8d per-ray model summed over the frame: hashtable 4*P1 + 4*P2 + 4*H; VCS 4*E + 4*L + 4*S + 4*H with S = 0
    (occupancy mask + popcount rank replaces the binary search); + 4 B per region-table entry read (int32 here, 8-byte
    pointers in the reference) + 3 B framebuffer write per pixel.  E counts the checks the kernel EXECUTES: iterations of the
    reference's EPSILON crawl that the kernel fast-forwards (DESIGN.md 3.2) move no bytes and are left out."""
    skipped = stats.get("crawl_skipped", 0)   # cluster-exists checks of fast-forwarded crawl iterations: counted (the reference executes them), never loaded
    if storage == "hashtable":
        b = 4 * stats["lookups"] + 4 * stats["table2_probes"] + 4 * stats["lookup_hits"]
    else:
        b = 4 * (stats["exist_checks"] - skipped) + 4 * stats["lookups"] + 4 * stats["lookup_hits"]
    return b + 4 * stats["region_reads"] + 3 * stats["rays"]


def ncu_summary(workload):
    """Figures of the dominant kernel from the committed ncu capture of this workload (profiles/ncu_summary.json): dram bytes and warp
    instructions per launch, threads per instruction, the kernel's name and the capture they come from.  {} when absent."""
    path = os.path.join(ROOT, "profiles", "ncu_summary.json")
    try:
        return dict(json.load(open(path)).get(workload, {}))
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------------------------------
def run_reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref host build of the unmodified
    reference; the C restatement only if that build is absent) on all host threads, same scene / camera / metric."""
    if rank != 0:
        return
    from oracle import pyoracle as po
    from voxelraymarcher_b200 import scenes
    kind = "refh" if po.available("refh") else "orc"
    cores = os.cpu_count() or 1
    xyz, rgb = scenes.terrain(SCENE_SIZE, SCENE_SEED)
    po.set_lighting(kind)
    ref = po.OracleScene(kind)
    ref.add_voxels(xyz, rgb)
    ref.build(STORAGE)
    cams = [po.make_camera(*_orbit_args(view_of(i, 0, 1)), kind) for i in range(args.warmup + args.steps)]   # the frames rank 0 renders at N = 1
    for i in range(args.warmup):
        ref.render(cams[i], WIDTH, HEIGHT, ALGORITHM, want_hits=False, threads=cores)
    t0 = time.perf_counter()
    for i in range(args.steps):
        last = ref.render(cams[args.warmup + i], WIDTH, HEIGHT, ALGORITHM, want_hits=False, threads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [last["rgb"]])
    value = WIDTH * HEIGHT * args.steps / dt / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference" if kind == "refh" else "port",
                         "sample": f"full {WIDTH}x{HEIGHT} frame per step, {args.steps} steps, traversal only (scene build excluded)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


DUMP_PIXELS = 1 << 21     # sampled pixels over all dumped frames: 2^21 x 12 B of colour + 2^21 / frames x 4 B of index <= 32 MiB


def dump_outputs(directory, frames):
    """--dump-outputs: the frames of the last timed step (one per rank, HxWx3 uint8) at a fixed, seeded sample of pixel positions
    (the same for every frame and every run), as float32 .npy files in `directory`:
        frame_rgb.npy          (frames, pixels, 3)  colour channels 0..255
        frame_pixel_index.npy  (pixels,)            row-major pixel index y * WIDTH + x (< 2^24: exact in float32)"""
    os.makedirs(directory, exist_ok=True)
    n = DUMP_PIXELS // len(frames)
    idx = np.sort(np.random.default_rng(20240101).choice(WIDTH * HEIGHT, n, replace=False))
    rgb = np.stack([np.asarray(f).reshape(WIDTH * HEIGHT, 3)[idx] for f in frames]).astype(np.float32)
    np.save(os.path.join(directory, "frame_rgb.npy"), rgb)
    np.save(os.path.join(directory, "frame_pixel_index.npy"), idx.astype(np.float32))


def _orbit_args(view):
    ang = np.float64(-0.75 * np.pi) + 2.0 * np.pi * (view % ORBIT_VIEWS) / ORBIT_VIEWS
    org = (float(np.float32(ORBIT_CENTRE[0] + ORBIT_RADIUS * np.cos(ang))), ORBIT_HEIGHT, float(np.float32(ORBIT_CENTRE[2] + ORBIT_RADIUS * np.sin(ang))))
    return org, ORBIT_CENTRE, (0.0, 1.0, 0.0), 60.0, np.float32(WIDTH) / np.float32(HEIGHT)


def workload_config():
    return {"workload": f"terrain{SCENE_SIZE}_4k_{STORAGE}_{ALGORITHM}", "scene": f"procedural {SCENE_SIZE}^3 terrain, seed {SCENE_SEED}, ~32 M voxels (BASELINE.json configs[2])",
            "resolution": f"{WIDTH}x{HEIGHT}", "storage": STORAGE, "algorithm": ALGORITHM, "shadows": True,
            "views": "one frame per GPU per step: (step k, rank r) renders view (25*k + r*64/N) mod 64 of a 64-view orbit of radius 498 at height 352 around (256,64,256); "
                     "view 0 = SURVEY.md 8d-3's camera (-96,352,-96), fov 60", "l2": "flushed between steps (512 MiB write, outside the per-step event pairs)",
            "parallelism": "frames sharded across GPUs (one per GPU per step, all different), structure replicated, frames stored into rank 0's buffer by the render kernels "
                           "(NVLink peer memory) + a completion word per rank; no collective on the data path"}


# ------------------------------------------------------------------------------------------------------------------
def build_bytes_model(n, unique, regions, diameter, storage):
    """Algorithmic HBM bytes of one structure build (DESIGN.md 3.1): what the kernels must read and write once.
    keys: 12 B xyz in + 4 B key out.  Stable LSD radix sort, 32-bit keys when 18 + log2(D^3) <= 32, 9-bit digits: per pass 4 B
    (histogram read) + 8 B in + 8 B out.  Dedupe + region heads: keep flags 4 in + 4 out, scan 4 in + 4 out, heads 8 in.
    VCS: 4 B key in + one 8 B header word per voxel + the zero-fill of the headers (64 KB per region); colours stay where the
    sort left them.  Hash table: 4 B (cluster mask) + 8 B (key, colour) in + 8 B slot out per voxel + the fill of both tables
    (2 x 1.25 x 8 B per voxel)."""
    key_bits = 18 + max(1, int(np.ceil(np.log2(max(2, diameter ** 3)))))
    key_bytes = 4 if key_bits <= 32 else 8
    passes = -(-key_bits // 9)
    per_voxel = (12 + key_bytes) + passes * (key_bytes + 2 * (key_bytes + 4)) + (8 + 8 + 8)
    b = n * per_voxel
    if storage == "vcs":
        b += unique * (4 + 8) + regions * 65536
    else:
        b += unique * (4 + 8 + 8) + 2 * (unique + unique // 4 + 2 * regions) * 8
    return int(b), passes


def timed_build(api, device, storage, voxels_on_gpu):
    """(scene, dict): generate the terrain on the GPU (vrm_scene_generate_terrain, identical voxel set to scenes.terrain: tested),
    build `storage`; event time of vrm_scene_build."""
    s = api.VoxelScene(device)
    n = s.generate_terrain(SCENE_SIZE, SCENE_SEED)
    s.synchronize()
    ms = s.generate_voxel_scene(storage)
    info = s.info()
    peak, _ = measured_peak()
    model, passes = build_bytes_model(n, info["unique_voxels"], info["filled"], info["diameter"], storage)
    gbs = model / (ms * 1e-3) / 1e9
    return s, {"ms": ms, "mvoxels_per_s": n / ms / 1e3, "voxels": n, "unique_voxels": info["unique_voxels"], "regions": info["filled"],
               "structure_bytes": info["bytes"],
               "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "algorithmic_bytes": model,
                            "bytes_per_voxel": model / n, "sort_passes": passes}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-baselines", action="store_true", help="skip the cpu_baseline / ref_gpu / orbit legs (profiling runs)")
    ap.add_argument("--single-view", action="store_true", help="every step renders view 0 (the named single view; profiling runs)")
    ap.add_argument("--orbit-only", action="store_true", help="only the strong-scaling leg (configs[3], the 2048^3 orbit); prints its dict (tuning runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the frames of the last timed step to DIR/*.npy (float32), "
                                                          "to compare the outputs of two builds run with the same arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.orbit_only:
        ap.error("--dump-outputs dumps the frames of the timed steps; --orbit-only has none")
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    # Libraries (NCCL's version banner, for one) write to fd 1; the contract is ONE JSON line on stdout, so everything
    # before the final print goes to stderr.
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    numa_cpus = bind_to_gpu_numa_node(local_rank)
    import torch
    import torch.distributed as dist
    from voxelraymarcher_b200 import api

    if not torch.cuda.is_available() or not api.device_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    if args.orbit_only:
        stream = torch.cuda.Stream(dev)
        torch.cuda.set_stream(stream)
        orbit = orbit_leg(api, torch, dist, dev, local_rank, rank, world, stream)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        os.dup2(saved_stdout, 1)
        if rank == 0:
            print(json.dumps({"orbit_2048_strong_scaling": orbit, "n_gpus": n_gpus}), flush=True)
        return

    # ---- scene: generated and built on the GPU, replicated per rank (deterministic) --------------------------------------
    warm = api.VoxelScene(local_rank)            # loads the CUDA modules and fills the memory pool: the timed build below is not a cold start
    warm.generate_terrain(64, SCENE_SEED)
    warm.generate_voxel_scene(STORAGE)
    warm.close()
    warm, _ = timed_build(api, local_rank, STORAGE, True)
    warm.close()
    scene, build = timed_build(api, local_rank, STORAGE, True)
    stream = torch.cuda.Stream(dev)          # a dedicated non-default stream: kernels, flushes, signals and events all live here
    torch.cuda.set_stream(stream)
    scene.set_stream(stream.cuda_stream)

    total = args.warmup + args.steps
    frame = torch.zeros((HEIGHT, WIDTH, 3), dtype=torch.uint8, device=dev)
    # Exchange step (N > 1): the finished frames arrive on rank 0.  Preferred form: FUSED into the render kernel -- every rank maps
    # rank 0's gather buffer through CUDA IPC and its kernel stores the frame straight into its slot over NVLink / NVSwitch
    # (coalesced 96-byte row segments); a release store of the step's sequence number into the rank's completion word follows
    # every frame, and rank 0 waits for the words once, at the end.  Fallback (no peer access): render locally + NCCL gather per step.
    ring = min(total, 32)                    # frame slots per rank in rank 0's buffer (the consumer of a real pipeline frees them in order)
    peer, exchange = None, "none"
    if world > 1:
        from voxelraymarcher_b200 import multigpu
        try:
            peer = multigpu.PeerFrameBuffer(world * ring, WIDTH, HEIGHT, local_rank)
            exchange = ("fused: render kernels store into rank 0's buffer over NVLink peer memory (CUDA IPC); completion = release store of a sequence number "
                        "behind every frame, waited for by rank 0 (no collective)")
        except Exception as exc:  # noqa: BLE001
            peer, exchange = None, f"nccl gather of frames (peer mapping failed: {exc})"
        flags = torch.tensor([1 if peer is not None else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        if int(flags.item()) == 0 and peer is not None:
            peer.close()
            peer, exchange = None, "nccl gather of frames (peer mapping failed on another rank)"
    if peer is not None:
        scene.set_completion_flag(peer.flag_ptr(rank), 1)
    gathered = [torch.zeros_like(frame) for _ in range(world)] if (world > 1 and rank == 0 and peer is None) else None
    wait_status = torch.zeros(1, dtype=torch.int32, device=dev)
    flush = torch.zeros(512 << 20, dtype=torch.uint8, device=dev)
    views = [0 if args.single_view else view_of(i, rank, world) for i in range(total)]
    cams = [orbit_camera(api, v) for v in views]

    def out_ptr(i):
        return peer.ptr_for(rank * ring + i % ring) if peer is not None else frame.data_ptr()

    def step(i, ev0, ev1, evk):
        flush.add_(1)                       # evict L2 (512 MiB > 126 MB), not timed
        ev0.record(stream)
        scene.render_device(WIDTH, HEIGHT, ALGORITHM, cams[i], out_ptr(i))
        evk.record(stream)
        if world > 1 and peer is None:
            dist.gather(frame, gathered, dst=0)
        if peer is not None and rank == 0 and i == total - 1:
            peer.wait_flags(stream.cuda_stream, total, timeout_ms=30000, d_status_ptr=wait_status.data_ptr())   # every rank's last frame has landed
        ev1.record(stream)

    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(total)]
    for i in range(args.warmup):
        step(i, *evs[i])
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)                          # let nvidia-smi come up: the timed region itself is only tens of milliseconds
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    wall0 = time.perf_counter()
    for i in range(args.warmup, total):
        step(i, *evs[i])
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    wall = time.perf_counter() - wall0
    step_ms = [evs[i][0].elapsed_time(evs[i][1]) for i in range(args.warmup, total)]
    kern_ms = [evs[i][0].elapsed_time(evs[i][2]) for i in range(args.warmup, total)]
    t_ms = float(sum(step_ms))
    tk_ms = float(sum(kern_ms))
    if int(wait_status.item()) != 0:
        raise SystemExit("bench.py: timed out waiting for the completion words of the other ranks")
    # the frames of the last timed step as rank 0 holds them (copied before later renders reuse `frame`)
    last_frames = None
    if args.dump_outputs and rank == 0 and peer is None:
        last_frames = [frame.cpu()] if world == 1 else [g.cpu() for g in gathered]

    exchange_ok = None
    if peer is not None:
        # outside the timed region: the gathered slots of the last two steps must equal local renders of the same cameras
        scene.set_completion_flag(None)
        dist.barrier()
        if rank == 0:
            full = peer.to_tensor()
            if args.dump_outputs:
                last_frames = [full[r * ring + (total - 1) % ring].cpu() for r in range(world)]
            exchange_ok = True
            for r in range(world):
                for i in (total - 2, total - 1):
                    scene.render_device(WIDTH, HEIGHT, ALGORITHM, orbit_camera(api, 0 if args.single_view else view_of(i, r, world)), frame.data_ptr())
                    torch.cuda.synchronize(dev)
                    exchange_ok = exchange_ok and bool(torch.equal(full[r * ring + i % ring], frame))
            del full
        dist.barrier()

    # ---- e2e: host-buffer C-ABI call (camera host -> device + frame D2H inside the timed region), pinned result buffer ---------
    host_frame = torch.zeros((HEIGHT, WIDTH, 3), dtype=torch.uint8).pin_memory()
    host_np = host_frame.numpy()
    e2e_s = 0.0
    if world > 1:
        dist.barrier()
    for i in range(total):
        flush.add_(1)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        scene.render(WIDTH, HEIGHT, ALGORITHM, cams[i], rgb_out=host_np)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            e2e_s += dt
    # the same call with a PAGEABLE caller buffer (what a plain C caller such as the CLI passes)
    pageable = np.zeros((HEIGHT, WIDTH, 3), np.uint8)
    pg_s = 0.0
    for i in range(total):
        flush.add_(1)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        scene.render(WIDTH, HEIGHT, ALGORITHM, cams[i], rgb_out=pageable)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            pg_s += dt
    clocks = sampler.stop() if rank == 0 else None

    if world > 1:
        red = torch.tensor([t_ms, tk_ms, e2e_s, pg_s], dtype=torch.float64, device=dev)
        dist.all_reduce(red, op=dist.ReduceOp.MAX)
        t_ms, tk_ms, e2e_s, pg_s = [float(v) for v in red.tolist()]

    rays_total = WIDTH * HEIGHT * args.steps * n_gpus
    value = rays_total / (t_ms * 1e-3) / 1e6
    value_no_gather = rays_total / (tk_ms * 1e-3) / 1e6
    e2e_value = rays_total / e2e_s / 1e6

    # ---- strong scaling of BASELINE.json configs[3]: the 64-view 1080p orbit of the 2048^3 scene, views claimed dynamically ----
    orbit = None
    if not args.no_baselines:
        orbit = orbit_leg(api, torch, dist, dev, local_rank, rank, world, stream)

    line = None
    if rank == 0:
        # ---- roofline of the dominant kernel (render): algorithmic bytes from the kernel's own event counters, summed over the
        # frames of the timed region (statistics build of the same kernel, outside the timed region) ---------------------------
        scene.set_statistics(True, as_executed=True)      # the work the timed kernels did (dead shadow rays are not traced)
        per_view = {}
        for v in sorted(set(views[args.warmup:])):
            scene.render_device(WIDTH, HEIGHT, ALGORITHM, orbit_camera(api, v), frame.data_ptr())
            scene.synchronize()
            per_view[v] = scene.get_statistics()
        scene.set_statistics(False)
        keys = ("exist_checks", "exist_false", "lookups", "lookup_hits", "table2_probes", "region_reads", "rays", "crawl_skipped")
        stats = {k: sum(per_view[v][k] for v in views[args.warmup:]) for k in keys}
        peak, peak_src = measured_peak()
        k_ms = float(np.mean(kern_ms))
        alg_bytes = algorithmic_bytes(stats, STORAGE) / args.steps
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9
        cfg = workload_config()
        if args.single_view:
            cfg["views"] = "every step renders view 0 (--single-view)"
        # the named single view (configs[2] as written), L2 flushed, median of 9
        times = []
        cam0 = orbit_camera(api, 0)
        for i in range(11):
            flush.add_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream); scene.render_device(WIDTH, HEIGHT, ALGORITHM, cam0, frame.data_ptr()); e1.record(stream)
            torch.cuda.synchronize(dev)
            if i >= 2:
                times.append(e0.elapsed_time(e1))
        sv_ms = float(np.median(times))
        # the roofs that bind: L2 (micro-benchmarked here: 8-byte gathers over an L2-resident working set) and instruction issue
        # (warp instructions of the committed ncu capture of the single view / (SMs x 4 schedulers x SM clock x kernel time))
        l2 = None
        try:
            l2 = api.microbench_l2(local_rank, 48 << 20)
        except Exception:  # noqa: BLE001
            pass
        summ = ncu_summary(cfg["workload"])
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        issue = None
        if summ.get("warp_instructions_per_launch"):
            wi = float(summ["warp_instructions_per_launch"])
            issue = {"warp_instructions_single_view": wi, "issue_frac": wi / (148 * 4 * sm_mhz * 1e6 * sv_ms * 1e-3), "threads_per_instruction": summ.get("threads_per_instruction"),
                     "source": summ.get("source")}
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": summ.get("dram_bytes_per_launch"),
                    "kernel": summ.get("kernel", "render kernel (VCS, longest axis)"), "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg_bytes,
                    "bytes_per_ray": alg_bytes / (WIDTH * HEIGHT), "peak_source": peak_src,
                    "binding_roof": "instruction issue (the touched working set is L1/L2-resident: DRAM traffic is ~1 % of the algorithmic bytes)",
                    "issue": issue,
                    "l2": None if l2 is None else {"gather8_gbs": l2["gather8_gbs"], "gather8_loads_per_ns": l2["gather8_loads_per_ns"], "stream_gbs": l2["stream_gbs"],
                                                   "working_set_bytes": l2["working_set_bytes"],
                                                   # every item of the byte model except the frame store is one load: loads per ns against the gather roof
                                                   "achieved_loads_per_ns": (alg_bytes - 3 * WIDTH * HEIGHT) / 4 / (k_ms * 1e6),
                                                   "frac_of_gather_roof": (alg_bytes - 3 * WIDTH * HEIGHT) / 4 / (k_ms * 1e6) / l2["gather8_loads_per_ns"] if l2["gather8_loads_per_ns"] else None},
                    "note": "SURVEY.md 8d per-ray model, with 4 B per region-table read (the table holds int32 here; the reference's 8-byte pointers would make it "
                            "+4 B per region read, ~+22 B per ray); traffic / issue figures come from the committed ncu capture of the single view (profiles/ncu_summary.json)"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 60, "d2h_bytes_per_step": WIDTH * HEIGHT * 3,
                    "pageable_caller_buffer": {"value": rays_total / pg_s / 1e6, "unit": UNIT}},
            "gpu_launches": launches_per_step(world, peer is not None) * args.steps,
            "roofline": roofline, "exchange": exchange, "exchange_verified": exchange_ok,
            "ms_per_frame_kernel": tk_ms / args.steps, "value_without_gather": value_no_gather, "wall_s_timed_region": wall,
            "single_view": {"ms_per_frame": sv_ms, "mrays_per_s": WIDTH * HEIGHT / sv_ms / 1e3, "camera": "(-96,352,-96) -> (256,64,256), fov 60 (SURVEY.md 8d-3)"},
            "views": views[args.warmup:], "kernel_ms_per_step": [round(x, 4) for x in kern_ms],
            "build": build, "numa_cpus": numa_cpus,
            "stats_per_ray": {k: stats[k] / stats["rays"] for k in ("exist_checks", "exist_false", "lookups", "lookup_hits", "region_reads", "crawl_skipped")},
        }
        if orbit is not None:
            line["orbit_2048_strong_scaling"] = orbit
        if n_gpus == 1 and not args.no_baselines:
            line.update(baseline_legs(api, scene, cam0, flush, dev))
    scene.close()
    if world > 1:
        dist.barrier()
        if peer is not None:
            peer.close()
        dist.destroy_process_group()
    if last_frames is not None:
        dump_outputs(args.dump_outputs, last_frames)
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    if rank == 0:
        print(json.dumps(line), flush=True)


def launches_per_step(world, fused):
    """Kernels of ours per step on every rank: the render kernel + the small kernel that continues its parked rays, + the
    completion-word store when the exchange is fused (N > 1)."""
    return 2 + (1 if (world > 1 and fused) else 0)


def orbit_views_2048(api, w, h):
    cams = []
    for v in range(64):
        ang = 2.0 * np.pi * (v + 0.37) / 64
        r, el = 1.5 * 1024.0, np.deg2rad(20.0)
        org = (float(1024 + r * np.cos(el) * np.cos(ang)), float(1024 + r * np.sin(el)), float(1024 + r * np.cos(el) * np.sin(ang)))
        cams.append(api.Camera(org, (1024.0, 1024.0, 1024.0), (0.0, 1.0, 0.0), 60.0, np.float32(w) / np.float32(h)))
    return cams


def orbit_leg(api, torch, dist, dev, local_rank, rank, world, stream):
    """BASELINE.json configs[3]: 2048^3 sparse scene (~36 M voxels, generated and built on every GPU), 64-view orbit at 1920x1080,
    VCS, both algorithms.  STRONG scaling: the 64 views are a fixed batch; ranks claim them dynamically from a counter in rank 0's
    buffer (multigpu.render_views_dynamic) and store them into rank 0's buffer; time = rank 0's clock from the barrier until all 64
    frames have landed, best of 3."""
    w, h = 1920, 1080
    try:
        s = api.VoxelScene(local_rank)
        n = s.generate_sparse_shells(2048, 64, 7, 35)
        build_ms = s.generate_voxel_scene("vcs")
        s.set_stream(stream.cuda_stream)
        cams = orbit_views_2048(api, w, h)
        out = {"views": 64, "resolution": f"{w}x{h}", "voxels": n, "build_ms": build_ms, "scaling": "strong", "assignment": "dynamic view claiming (atomic counter in rank 0's buffer)" if world > 1 else "one GPU"}
        claim_stream = torch.cuda.Stream(dev)
        peer = None
        if world > 1:
            from voxelraymarcher_b200 import multigpu
            peer = multigpu.PeerFrameBuffer(64, w, h, local_rank)
        else:
            frames = torch.zeros((64, h, w, 3), dtype=torch.uint8, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        for algo in ("longestaxis", "original"):
            best, counts = None, None
            for rep in range(4):
                torch.cuda.synchronize(dev)
                if world > 1:
                    if rank == 0:
                        peer.reset_counters()
                    dist.barrier()
                    torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                if world > 1:
                    mine = multigpu.render_views_dynamic(s, peer, cams, w, h, algo, stream, claim_stream)
                    if rank == 0:
                        peer.wait_counter(stream.cuda_stream, 64, timeout_ms=60000, d_status_ptr=status.data_ptr())
                        torch.cuda.synchronize(dev)
                else:
                    for v in range(64):
                        s.render_device(w, h, algo, cams[v], frames[v].data_ptr())
                    torch.cuda.synchronize(dev)
                    mine = 64
                dt = (time.perf_counter() - t0) * 1e3
                if world > 1:
                    red = torch.tensor([dt], dtype=torch.float64, device=dev)
                    dist.all_reduce(red, op=dist.ReduceOp.MAX)
                    dt = float(red.item())
                    c = torch.zeros(world, dtype=torch.int32, device=dev)
                    c[rank] = mine
                    dist.all_reduce(c)
                    mine = c.tolist()
                if rep >= 1 and (best is None or dt < best):
                    best, counts = dt, mine
            out[algo] = {"ms_per_orbit": best, "mrays_per_s": 64 * w * h / best / 1e3, "views_per_rank": counts}
        if int(status.item()) != 0:
            out["error"] = "timed out waiting for frames"
        if world > 1:
            dist.barrier()
            peer.close()
        s.close()
        return out
    except Exception as exc:  # noqa: BLE001
        return {"error": f"{type(exc).__name__}: {exc}"}


def baseline_legs(api, scene, cam, flush, dev):
    """Baselines timed in the same run (north star): the reference's own CUDA kernels rebuilt for sm_100a on this GPU, and
    the reference's traversal built for the host cores.  Reported, never the thing measured.  Also times the other three
    storage x algorithm combinations of the native path on the same frame (the named single view) and the hash-table build."""
    import torch
    from oracle import pyoracle as po
    from voxelraymarcher_b200 import scenes
    out = {}
    cores = os.cpu_count() or 1
    xyz, rgb = scenes.terrain(SCENE_SIZE, SCENE_SEED)     # host copy of the voxel list for the reference builds
    # native: all four combinations, median of 7 launches, L2 flushed
    combos = {}
    scenes_by_storage = {STORAGE: scene}
    builds = {}
    for storage in ("vcs", "hashtable"):
        if storage not in scenes_by_storage:
            warm = api.VoxelScene(scene.device)      # first use of this storage's builder kernels / allocations: not part of the timed build
            warm.generate_terrain(64, SCENE_SEED)
            warm.generate_voxel_scene(storage)
            warm.close()
            warm, _ = timed_build(api, scene.device, storage, True)
            warm.close()
            s, builds[storage] = timed_build(api, scene.device, storage, True)
            scenes_by_storage[storage] = s
        s = scenes_by_storage[storage]
        fb = torch.zeros((HEIGHT, WIDTH, 3), dtype=torch.uint8, device=dev)
        cur = torch.cuda.current_stream(dev)
        s.set_stream(cur.cuda_stream)
        for algo in ("longestaxis", "original"):
            times = []
            for i in range(9):
                flush.add_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(cur); s.render_device(WIDTH, HEIGHT, algo, cam, fb.data_ptr()); e1.record(cur)
                torch.cuda.synchronize(dev)
                if i >= 2:
                    times.append(e0.elapsed_time(e1))
            ms = float(np.median(times))
            combos[f"{storage}+{algo}"] = {"ms_per_frame": ms, "mrays_per_s": WIDTH * HEIGHT / ms / 1e3, "build_ms": s.build_ms}
    out["build_hashtable"] = builds.get("hashtable")
    # reference CUDA kernels (default nvcc flags) on the same frame
    if po.available("refg"):
        po.set_lighting("refg")
        for storage in ("vcs", "hashtable"):
            ref = po.OracleScene("refg")
            t0 = time.perf_counter()
            ref.add_voxels(xyz, rgb)
            ref.build(storage)
            host_build_s = time.perf_counter() - t0
            for algo in ("longestaxis", "original"):
                ms = np.zeros(5, np.float32)
                rc = ref.lib.refg_render_timed(ref.h, po._ptr(cam.data), po._ptr(np.zeros(3, np.float32)), 1, po.ALGORITHM[algo], WIDTH, HEIGHT, 2, 5, po._ptr(ms))
                if rc == 0:
                    m = float(np.median(ms))
                    c = combos[f"{storage}+{algo}"]
                    c.update(ref_gpu_ms_per_frame=m, ref_gpu_mrays_per_s=WIDTH * HEIGHT / m / 1e3, speedup_vs_ref_gpu=m / c["ms_per_frame"], ref_host_build_s=host_build_s)
            ref.close()
    out["combos"] = combos
    # reference traversal on the host cores (cpu_baseline)
    kind = "refh" if po.available("refh") else "orc"
    po.set_lighting(kind)
    ref = po.OracleScene(kind)
    ref.add_voxels(xyz, rgb)
    ref.build(STORAGE)
    ref.render(cam.data, WIDTH, HEIGHT, ALGORITHM, want_hits=False, threads=cores)
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        ref.render(cam.data, WIDTH, HEIGHT, ALGORITHM, want_hits=False, threads=cores)
    dt = time.perf_counter() - t0
    ref.close()
    out["cpu_baseline"] = {"value": WIDTH * HEIGHT * reps / dt / 1e6, "unit": UNIT, "cores": cores, "kind": "reference" if kind == "refh" else "port",
                           "sample": f"{reps} full {WIDTH}x{HEIGHT} frames of the same scene/camera, traversal only (scene build excluded)"}
    for s in scenes_by_storage.values():
        if s is not scene:
            s.close()
    return out


if __name__ == "__main__":
    main()
