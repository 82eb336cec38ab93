"""GPU tier: the scene builder (csrc/vrm_build.cu) at its edges, against a last-insert-wins model of the staged list.

The builder sorts 32- or 64-bit keys (regionCell << 18 | cluster << 9 | code) with its own LSD radix sort (2048-key tiles, digits of
up to 9 bits, so passes = ceil(keyBits / 9) with keyBits = 18 + ceil(log2 D^3)), dedupes last-write-wins, and fills the VCS tables or
inserts into per-region cuckoo tables that are re-seeded and rebuilt when they fail.  Every case below names the path it reaches.
A built scene must hold exactly the model's voxels -- info(), read_voxels(), lookup of every stored voxel and of misses -- for both
storage types and, where the oracle's region table stays small, trace bit-exactly like the oracle (oracle/vrm_oracle.c).

A build that fails must leave the staged scene as it was: the last case stages 531 441 one-voxel regions, which exceed the VCS index
widths after the sort, and then builds the same handle as a hash table."""
import math
import re

import numpy as np
import pytest

from tests.common import build_oracle, oracle_kind, po
from voxelraymarcher_b200 import api

pytestmark = pytest.mark.gpu

STORAGES = ["hashtable", "vcs"]
ERR_INVALID, ERR_STATE = 1, 3


# ---- the model -------------------------------------------------------------------------------------------------------------------------
def coord_key(xyz):
    """int64 key ordered like (x, y, z) for |c| < 2^20."""
    k = np.asarray(xyz, np.int64) + (1 << 20)
    return (k[:, 0] << 42) | (k[:, 1] << 21) | k[:, 2]


def model(xyz, rgb):
    """The staged list in call order -> (xyz, rgb) of the last-insert-wins set sorted by (x, y, z), and the info() it builds to."""
    xyz = np.asarray(xyz, np.int32).reshape(-1, 3)
    rgb = np.asarray(rgb, np.uint32).reshape(-1)
    n = len(rgb)
    if n:
        keys = coord_key(xyz)
        _, first_rev = np.unique(keys[::-1], return_index=True)   # first in the reversed list = last insert
        last = n - 1 - first_rev
        mx, mr = xyz[last], rgb[last]
        reg = np.floor_divide(xyz, 64)
        lo, hi = min(0, int(reg.min())), max(0, int(reg.max()))
        filled = len(np.unique(coord_key(reg)))
    else:
        mx, mr = np.zeros((0, 3), np.int32), np.zeros(0, np.uint32)
        lo = hi = 0
        filled = 0
    info = dict(diameter=hi - lo + 1, min_coord=lo, filled=filled, unique_voxels=len(mr))
    return mx, mr, info


def key_bits(d):
    return 18 + math.ceil(math.log2(d ** 3)) if d > 1 else 18


def passes(d):
    return -(-key_bits(d) // 9)


# ---- the shared check ------------------------------------------------------------------------------------------------------------------
def miss_queries(s, mx, rng, max_neighbours=200_000):
    """Cells that hold no voxel: unstored face neighbours of stored voxels, random cells inside the table, cells one past each face of
    scene_box(), and coordinates near +-2^23 (the last two lie outside the region table)."""
    (o, d) = [np.asarray(v, np.int64) for v in s.scene_box()]
    inside = []
    if len(mx):
        base = mx if len(mx) <= max_neighbours else mx[rng.choice(len(mx), max_neighbours, replace=False)]
        for a in range(3):
            for step in (-1, 1):
                nb = base.astype(np.int64).copy()
                nb[:, a] += step
                inside.append(nb)
    inside.append(o + rng.integers(0, d, size=(20_000, 3)))
    inside = np.concatenate(inside)
    stored = coord_key(mx) if len(mx) else np.zeros(0, np.int64)
    inside = inside[~np.isin(coord_key(inside), stored)]
    outside = []
    for a in range(3):
        for edge in (o[a] - 1, o[a] + d[a]):
            p = o + rng.integers(0, d, size=(500, 3))
            p[:, a] = edge
            outside.append(p)
    big = (1 << 23) - 1
    outside.append(np.array([[big, 0, 0], [-big, 0, 0], [0, big, 0], [0, -big, 0], [0, 0, big], [0, 0, -big],
                             [big, big, big], [-big, -big, -big], [big - 70, 5, -big + 3]], np.int64))
    return inside.astype(np.int32), np.concatenate(outside).astype(np.int32)


def check_scene(s, mx, mr, info, seed=0):
    """info(), read_voxels(), count_voxels() and lookup of stored voxels and of misses against the model."""
    got = s.info()
    assert {k: got[k] for k in info} == info, (got, info)
    gx, gr = s.read_voxels()
    assert gx.shape == mx.shape and np.array_equal(gx, mx), (len(gx), len(mx))
    assert np.array_equal(gr, mr)
    assert s.count_voxels() == len(mr)
    if len(mx):
        col, ex = s.lookup(mx)
        assert np.array_equal(col, mr) and ex.all()
    inside, outside = miss_queries(s, mx, np.random.default_rng(seed))
    col, _ = s.lookup(inside)
    assert (col == api.EMPTY).all(), inside[col != api.EMPTY][:5]
    col, ex = s.lookup(outside)
    assert (col == api.EMPTY).all() and not ex.any(), outside[(col != api.EMPTY) | (ex != 0)][:5]


def aimed_rays(mx, n, rng, dist=(20.0, 150.0)):
    """Rays from random points around stored voxels, aimed at them: most hit something near the target."""
    t = mx[rng.integers(0, len(mx), n)].astype(np.float64) + rng.uniform(0.2, 0.8, (n, 3))
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o = t + d * rng.uniform(*dist, (n, 1))
    return np.concatenate([o, -d], 1).astype(np.float32)


def check_against_oracle(s, xyz, rgb, storage, rays):
    kind = oracle_kind()
    po.set_lighting(kind)
    ref = build_oracle(kind, xyz, rgb, storage)
    try:
        rinfo, info = ref.info(), s.info()
        assert (rinfo["diameter"], rinfo["min_coord"], rinfo["filled"]) == (info["diameter"], info["min_coord"], info["filled"])
        for algo in ("original", "longestaxis"):
            want = ref.trace_rays(rays, algo)
            got = s.trace_rays(rays, algo, want_hits=True)
            assert np.array_equal(got["hits"], want["hits"]), (storage, algo, int((got["hits"] != want["hits"]).any(1).sum()))
            assert np.array_equal(got["colour"], want["colour"]), (storage, algo)
            assert want["hits"][:, 3].sum() > len(rays) // 4   # the rays do reach voxels
    finally:
        ref.close()


def build_and_check(xyz, rgb, storage, seed=0, oracle_rays=2000):
    mx, mr, info = model(xyz, rgb)
    s = api.VoxelScene(0)
    s.add_voxels(xyz, rgb)
    s.generate_voxel_scene(storage)
    check_scene(s, mx, mr, info, seed)
    if oracle_rays and len(mx) and info["diameter"] <= 100:
        check_against_oracle(s, xyz, rgb, storage, aimed_rays(mx, oracle_rays, np.random.default_rng(seed + 1)))
    return s, info


def with_duplicates(xyz, rgb, frac, rng):
    """The list plus re-inserts of about frac of its voxels with new colours, all shuffled together."""
    k = int(len(rgb) * frac)
    pick = rng.integers(0, len(rgb), k)
    xyz = np.concatenate([xyz, xyz[pick]])
    rgb = np.concatenate([rgb, rng.integers(0, 1 << 24, k, dtype=np.uint32)])
    order = rng.permutation(len(rgb))
    return xyz[order], rgb[order]


def colours(rng, n):
    return rng.integers(0, 1 << 24, n, dtype=np.uint32)


# ---- tile and scan boundaries ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("dups", [False, True], ids=["unique", "dups"])
@pytest.mark.parametrize("n", [1, 2, 2047, 2048, 2049, 6145, 2048 * 2048 + 1])
def test_tile_and_scan_boundaries(n, dups, storage):
    """n around the 2048-key sort tile: a partial last tile (2047, 2049, 6145), exactly one tile, one and two voxels.  Small n with a
    3^3 region table takes the separate sort-scratch allocation, large n carves it out of the xyz staging array; 2048^2 + 1 voxels
    make the scan over n recurse to its third level (2049 tile sums).  The duplicate variant re-inserts ~30 % (the keep_last /
    compaction path)."""
    rng = np.random.default_rng(n + dups)
    if n < 100_000:
        flat = rng.choice(150 ** 3, size=n, replace=False)       # coordinates in [-100, 50): regions -2 .. 0, D = 3
        xyz = (np.stack(np.unravel_index(flat, (150,) * 3), 1) - 100).astype(np.int32)
    else:
        # spread thin (~400 voxels per region, D = 22, still 32-bit keys): dense random subsets of a region defeat the cuckoo hashing
        cand = rng.integers(-700, 700, (n + n // 50, 3))
        _, first = np.unique(coord_key(cand), return_index=True)
        xyz = cand[np.sort(first)[:n]].astype(np.int32)
        assert len(xyz) == n
    rgb = colours(rng, n)
    if dups:
        keep = max(1, int(n * 0.7))
        xyz, rgb = with_duplicates(xyz[:keep], rgb[:keep], (n - keep) / keep, rng)
    build_and_check(xyz, rgb, storage, seed=n, oracle_rays=2000 if n > 2 else 0)


# ---- key width and pass parity ---------------------------------------------------------------------------------------------------------
KEY_CASES = {1: (18, 2), 2: (21, 3), 25: (32, 4), 26: (33, 4), 100: (38, 5), 1024: (48, 6)}


def extreme_scene(D, rng, cloud=5000):
    """Voxels in the region range [lo, lo + D) on every axis, with lo <= 0 < lo + D: the eight corner regions (with the corner voxels
    of each) plus a random cloud over the whole table."""
    lo = -(D // 2)
    hi = lo + D - 1
    pts = []
    for cx in (lo, hi):
        for cy in (lo, hi):
            for cz in (lo, hi):
                base = np.array([cx, cy, cz], np.int64) * 64
                local = np.concatenate([rng.integers(0, 64, (40, 3)), np.array([[0, 0, 0], [63, 63, 63], [0, 63, 0], [63, 0, 63]])])
                pts.append(base + local)
    pts.append(rng.integers(lo * 64, (hi + 1) * 64, (cloud, 3)))
    xyz = np.unique(np.concatenate(pts), axis=0)
    xyz = xyz[rng.permutation(len(xyz))].astype(np.int32)
    return xyz, colours(rng, len(xyz))


@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("dups", [False, True], ids=["unique", "dups"])
@pytest.mark.parametrize("D", sorted(KEY_CASES))
def test_key_width_and_pass_parity(D, dups, storage):
    """D = 1: 18 key bits, 2 passes.  D = 2: 21 bits, 3 passes.  D = 25: 32 bits, the last 32-bit key, 4 passes.  D = 26: 33 bits, the
    first 64-bit key.  D = 100: 38 bits, 5 passes.  D = 1024: 48 bits, 6 passes (and the first 48-bit key of read_voxels' sort).  An even
    pass count leaves the colours in the staging array, which the VCS then takes over without a copy (when there are no duplicates);
    an odd count, or a compaction, takes the copy."""
    assert (key_bits(D), passes(D)) == KEY_CASES[D]
    rng = np.random.default_rng(D * 2 + dups)
    xyz, rgb = extreme_scene(D, rng)
    if dups:
        xyz, rgb = with_duplicates(xyz, rgb, 0.3, rng)
    s, info = build_and_check(xyz, rgb, storage, seed=D)
    assert info["diameter"] == D
    if D == 1024:
        # the oracle's region table is a calloc of D^3 pointers (8 GiB virtual): only a small ray set near the populated low corner
        mx, _, _ = model(xyz, rgb)
        corner = mx[(mx < -(D // 2) * 64 + 64).all(1)]
        check_against_oracle(s, xyz, rgb, storage, aimed_rays(corner, 300, np.random.default_rng(5), dist=(5.0, 40.0)))


# ---- extent limit ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("storage", STORAGES)
def test_extent_limit(storage):
    """The region table always contains region 0: x = 65535 (regions 0 .. 1023) and x = -65472 (-1023 .. 0) give D = 1024 and build;
    x = 65536, x = -65473 and a span of -32768 .. 32768 give D = 1025 and are rejected (VRM_ERR_INVALID) before the staged voxels are
    touched -- the same handle rejects again and, once rebuilt without the offending voxel, builds."""
    lib = api.load_library()
    near = np.array([[1, 2, 3], [40, 7, 9]], np.int32)     # region 0 on every axis: the extent is one range over all three axes
    for edge in (65535, -65472):
        xyz = np.concatenate([near, [[edge, 5, 6]]]).astype(np.int32)
        s, info = build_and_check(xyz, np.arange(1, 4, dtype=np.uint32), storage, oracle_rays=0)
        assert info["diameter"] == 1024
    for bad in ([[65536, 0, 0]], [[-65473, 0, 0]], [[0, -32768, 0], [0, 32768, 0]]):
        xyz = np.concatenate([near, bad]).astype(np.int32)
        rgb = np.arange(1, len(xyz) + 1, dtype=np.uint32)
        s = api.VoxelScene(0)
        s.add_voxels(xyz, rgb)
        for _ in range(2):
            assert lib.vrm_scene_build(s.h, api.STORAGE[storage], None) == ERR_INVALID
            assert b"1024" in lib.vrm_last_error(s.h)
        s.close()


# ---- duplicate runs --------------------------------------------------------------------------------------------------------------------
HOT_RUN = 3 * 2048 + 5


def staged_calls(D, rng):
    """One coordinate staged HOT_RUN times with distinct colours, interleaved with other voxels, spread over add_voxels,
    add_voxels_device, insert_voxel and add_dense.  Returns the calls and the list they stage, in call order."""
    lo = -(D // 2)
    span = (lo * 64, (lo + D) * 64)
    hot = np.array([lo * 64 + 17, (lo + D) * 64 - 3, 3], np.int32)   # the dense boxes around it stay inside the table
    calls, xs, cs = [], [], []
    colour = iter(range(1, 1 << 30))
    remaining = HOT_RUN - 4                                             # the four add_dense calls stage it once each
    for kind in ["host", "device", "insert", "dense"] * 4 + ["host"]:
        if kind == "dense":
            origin = hot - np.array([3, 2, 4], np.int32)
            vol = np.full((7, 5, 9), api.EMPTY, np.uint32)
            cells = rng.choice(vol.size, vol.size // 3, replace=False)
            vol.reshape(-1)[cells] = [next(colour) for _ in cells]
            vol[3, 2, 4] = next(colour)                              # the hot cell, once per call (C order decides its place)
            xs.append((np.argwhere(vol != api.EMPTY) + origin).astype(np.int32))
            cs.append(vol[vol != api.EMPTY])
            calls.append(("dense", vol, origin))
            continue
        k = remaining if len(calls) == 16 else min(remaining, int(rng.integers(1, 40 if kind == "insert" else 1500)))
        remaining -= k
        x = np.concatenate([np.repeat(hot[None], k, 0), rng.integers(span[0], span[1], (2 * k + 1, 3)).astype(np.int32)])
        x = x[rng.permutation(len(x))]
        c = np.array([next(colour) for _ in range(len(x))], np.uint32)
        xs.append(x)
        cs.append(c)
        calls.append((kind, x, c))
    xyz, rgb = np.concatenate(xs), np.concatenate(cs)
    assert remaining == 0 and (coord_key(xyz) == coord_key(hot[None])[0]).sum() == HOT_RUN
    return calls, xyz, rgb


def stage(s, calls):
    import torch
    for kind, a, b in calls:
        if kind == "host":
            s.add_voxels(a, b)
        elif kind == "device":
            dx = torch.from_numpy(np.ascontiguousarray(a)).cuda()
            dr = torch.from_numpy(np.ascontiguousarray(b).view(np.int32)).cuda()
            torch.cuda.synchronize()
            s.add_voxels_device(dx.data_ptr(), dr.data_ptr(), len(b))
            s.synchronize()
        elif kind == "insert":
            for p, c in zip(a.tolist(), b.tolist()):
                s.insert_voxel(*p, c)
        else:
            s.add_dense(a, tuple(int(v) for v in b))


@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("D", [2, 26])
def test_duplicate_runs(D, storage):
    """A duplicate run longer than three sort tiles (3 * 2048 + 5 inserts of one coordinate) must keep its LAST colour: the radix
    sort has to be stable across tiles and calls of every kind, keep_last must flag the run's end, and the compaction must drop the
    rest -- with 32-bit keys (D = 2, 21 bits) and 64-bit keys (D = 26, 33 bits).  Then every coordinate staged two to four times in
    shuffled order."""
    rng = np.random.default_rng(D)
    calls, xyz, rgb = staged_calls(D, rng)
    mx, mr, info = model(xyz, rgb)
    assert info["diameter"] == D
    s = api.VoxelScene(0)
    stage(s, calls)
    s.generate_voxel_scene(storage)
    check_scene(s, mx, mr, info, seed=D)
    if D <= 100:
        check_against_oracle(s, xyz, rgb, storage, aimed_rays(mx, 2000, np.random.default_rng(D + 7)))
    # every coordinate duplicated, shuffled
    lo = -(D // 2)
    base = np.unique(rng.integers(lo * 64, (lo + D) * 64, (20_000, 3)), axis=0).astype(np.int32)
    reps = rng.integers(2, 5, len(base))
    xyz = np.repeat(base, reps, 0)
    order = rng.permutation(len(xyz))
    xyz = xyz[order]
    rgb = rng.permutation(len(xyz)).astype(np.uint32) + 1
    build_and_check(xyz, rgb, storage, seed=D + 1)


# ---- cuckoo rebuild --------------------------------------------------------------------------------------------------------------------
# vrm_build.cu seed_for / table_slots and vrm_core.cuh hash_key / hash_slot1 / hash_slot2, restated
M32 = 0xFFFFFFFF


def seed_for(ri, attempt, which):
    h = (ri * 0x9E3779B1 + attempt * 0x85EBCA77 + which * 0xC2B2AE3D + 0x27D4EB2F) & M32
    h ^= h >> 15
    h = (h * 0x2C1B3C6D) & M32
    h ^= h >> 12
    h = (h * 0x297A2D39) & M32
    h ^= h >> 15
    return h | 1


def table_slots(cnt):
    return cnt + cnt // 4 + 2


def hash_key(x, y, z):
    return (np.asarray(x, np.uint64) << 14) | (np.asarray(y, np.uint64) << 7) | np.asarray(z, np.uint64)


def hash_slot(key, seed, n):
    """mulhi32((key + 1) * seed, n), for slot 1 and slot 2 alike."""
    return ((((np.asarray(key, np.uint64) + 1) * np.uint64(seed)) & np.uint64(M32)) * np.uint64(n)) >> np.uint64(32)


def fits(keys, ri, attempt):
    """A placement of every key in its slot of table 1 or table 2 exists under the attempt's seeds (maximum bipartite matching)."""
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import maximum_bipartite_matching
    n = table_slots(len(keys))
    s1 = hash_slot(keys, seed_for(ri, attempt, 1), n).astype(np.int64)
    s2 = hash_slot(keys, seed_for(ri, attempt, 2), n).astype(np.int64) + n
    rows = np.repeat(np.arange(len(keys)), 2)
    g = csr_matrix((np.ones(2 * len(keys)), (rows, np.stack([s1, s2], 1).reshape(-1))), shape=(len(keys), 2 * n))
    return bool((maximum_bipartite_matching(g, perm_type="column") >= 0).all())


ALL_LOCAL = np.stack(np.unravel_index(np.arange(64 ** 3), (64,) * 3), 1)
ALL_KEYS = hash_key(ALL_LOCAL[:, 0], ALL_LOCAL[:, 1], ALL_LOCAL[:, 2])


def colliding_triple(ri, fail_attempts, rng):
    """Three region-local voxels whose keys share slot 1 AND slot 2 under the seeds of every attempt in fail_attempts (three keys on two
    slots cannot be placed: the region fails), and that fit under the seeds of the next attempt."""
    n = table_slots(3)
    tup = np.zeros(len(ALL_KEYS), np.int64)
    for a in fail_attempts:
        tup = tup * (n * n) + hash_slot(ALL_KEYS, seed_for(ri, a, 1), n).astype(np.int64) * n + hash_slot(ALL_KEYS, seed_for(ri, a, 2), n).astype(np.int64)
    order = np.argsort(tup, kind="stable")
    st = tup[order]
    bounds = np.flatnonzero(np.diff(st)) + 1
    groups = [g for g in np.split(order, bounds) if len(g) >= 3]
    nxt = max(fail_attempts) + 1
    for gi in rng.permutation(len(groups)):
        g = groups[gi]
        for _ in range(20):
            pick = rng.choice(g, 3, replace=False)
            if fits(ALL_KEYS[pick], ri, nxt):
                return ALL_LOCAL[pick]
    raise AssertionError(f"no colliding triple for region {ri}")


@pytest.mark.parametrize("fail_attempts", [(0,), (0, 1, 2)], ids=["fails-once", "fails-three-times"])
def test_cuckoo_rebuild(monkeypatch, capfd, fail_attempts):
    """Three-voxel regions (5 slots per table) whose keys collide in both tables under the seeds of attempt 0 (or of attempts 0, 1
    and 2) must fail their insertion round, be cleared, re-seeded, marked for retry and re-inserted; with three failing rounds the
    fourth runs in the second batch of three rounds the host launches.  Next to them small ordinary regions, which fit at attempt 0.
    The stderr trace (VRM_BUILD_TRACE=1) must report exactly that many failed regions per round -- this also catches a change of the
    hash functions that would let the test pass without reaching the path."""
    rng = np.random.default_rng(len(fail_attempts))
    D = 6
    cells = rng.permutation(D ** 3)[:60]                      # occupied region cells, ux + uy * D + uz * D^2
    bad = set(cells[:8].tolist())
    dense_index = {c: i for i, c in enumerate(sorted(cells.tolist()))}   # the dense region index: rank among the occupied cells
    xs = []
    for c in cells.tolist():
        ri = dense_index[c]
        rx, ry, rz = c % D, c // D % D, c // (D * D)
        if c in bad:
            local = colliding_triple(ri, fail_attempts, rng)
        else:
            while True:
                k = int(rng.integers(1, 40))
                local = ALL_LOCAL[rng.choice(len(ALL_LOCAL), k, replace=False)]
                if fits(hash_key(local[:, 0], local[:, 1], local[:, 2]), ri, 0):
                    break
        xs.append(local + 64 * np.array([rx, ry, rz]))
    xyz = np.concatenate(xs).astype(np.int32)
    xyz = xyz[rng.permutation(len(xyz))]
    rgb = colours(rng, len(xyz))
    mx, mr, info = model(xyz, rgb)
    assert info["diameter"] == D and info["filled"] == 60

    monkeypatch.setenv("VRM_BUILD_TRACE", "1")
    capfd.readouterr()
    s = api.VoxelScene(0)
    s.add_voxels(xyz, rgb)
    s.generate_voxel_scene("hashtable")
    err = capfd.readouterr().err
    rounds = [(int(r), int(f)) for r, f in re.findall(r"cuckoo round (\d+): (\d+) regions failed", err)]
    starts = [i for i, (r, _) in enumerate(rounds) if r == 0]
    assert starts, err
    last = [f for _, f in rounds[starts[-1]:]]
    # rounds run in batches of three; the round after the last failing one must run, so the last report covers whole batches up to it
    want = [len(bad) if r in fail_attempts else 0 for r in range(3 * -(-(max(fail_attempts) + 2) // 3))]
    assert last == want, (last, want)
    check_scene(s, mx, mr, info)
    check_against_oracle(s, xyz, rgb, "hashtable", aimed_rays(mx, 2000, np.random.default_rng(3)))


# ---- full and tiny regions -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("storage", STORAGES)
def test_full_and_tiny_regions(storage):
    """One full 64^3 region (every occupancy word all ones: vcs_fill gathers 32 voxels per word; one cuckoo region of 327 682 slots per
    table), single-voxel regions (3 slots per table), and colours 0 and >= 0x80000000 (the VCS keeps its cluster-exists flag in the
    top bit of the header's index word, never in a colour)."""
    rng = np.random.default_rng(11)
    full = ALL_LOCAL.astype(np.int32) + np.array([64, -64, 0], np.int32)
    singles = (np.array([[-2, 1, 1], [1, 1, -2], [0, 2, 0], [-1, -1, -1], [2, -2, 2]]) * 64 + rng.integers(0, 64, (5, 3))).astype(np.int32)
    xyz = np.concatenate([full, singles])
    rgb = colours(rng, len(xyz))
    rgb[:: 7] = 0
    rgb[3:: 11] = 0x80000000
    rgb[5:: 13] = 0xFFFFFFFF
    rgb[-5:] = [0, 0x80000000, 0xFFFFFFFF, 0x80000001, 0xC0000000]
    order = rng.permutation(len(xyz))
    xyz, rgb = xyz[order], rgb[order]
    _, _, info = model(xyz, rgb)
    assert info["filled"] == 6 and info["unique_voxels"] == 64 ** 3 + 5
    build_and_check(xyz, rgb, storage, seed=11)


# ---- a failed build --------------------------------------------------------------------------------------------------------------------
def one_voxel_per_region(rng, D=81):
    """D^3 regions with one voxel each, shuffled: 531 441 regions exceed the VCS index widths (>= 524 288), after the sort.  D = 81:
    38 key bits, 64-bit keys, 5 passes, so the staged colour array holds a sort pass's output when the check fails."""
    cells = np.stack(np.unravel_index(np.arange(D ** 3), (D,) * 3), 1)
    xyz = (cells * 64 + rng.integers(0, 64, cells.shape)).astype(np.int32)
    order = rng.permutation(len(xyz))
    return xyz[order], colours(rng, len(xyz))


@pytest.mark.parametrize("variant", ["plain", "add-after", "duplicates"])
def test_failed_build_leaves_the_staged_scene(variant):
    """A VCS build that fails (VRM_ERR_INVALID: too many regions for its index widths) after the sort consumed the staging arrays must
    leave the handle as if it had not been attempted: the hash-table build of the same handle holds the model's scene.  Variants: voxels
    added after the failure (recolouring staged coordinates and new ones) still win; a staged list with duplicates fails after the
    compaction."""
    rng = np.random.default_rng(81)
    xyz, rgb = one_voxel_per_region(rng)
    if variant == "duplicates":
        xyz, rgb = with_duplicates(xyz, rgb, 0.1, rng)
    assert passes(81) == 5
    lib = api.load_library()
    s = api.VoxelScene(0)
    s.add_voxels(xyz, rgb)
    for _ in range(2):                                          # the retry fails the same way: the staged scene is unchanged
        assert lib.vrm_scene_build(s.h, api.STORAGE_VCS, None) == ERR_INVALID
        assert b"index widths" in lib.vrm_last_error(s.h)
    with pytest.raises(api.VrmError):
        s.info()
    if variant == "add-after":
        pick = rng.choice(len(xyz), 5000, replace=False)
        fresh = xyz[pick[:100]].copy()                           # new voxels next to staged ones, in the same regions
        fresh[:, 2] = (fresh[:, 2] & ~63) | ((fresh[:, 2] + 1) & 63)
        more = np.concatenate([xyz[pick], fresh])
        more_rgb = colours(rng, len(more))
        s.add_voxels(more, more_rgb)
        for p, c in zip(xyz[pick[:10]].tolist(), range(10)):
            s.insert_voxel(*p, 0xABC000 + c)
        xyz = np.concatenate([xyz, more, xyz[pick[:10]]])
        rgb = np.concatenate([rgb, more_rgb, np.arange(10, dtype=np.uint32) + 0xABC000])
    mx, mr, info = model(xyz, rgb)
    s.generate_voxel_scene("hashtable")
    check_scene(s, mx, mr, info, seed=81)
    check_against_oracle(s, xyz, rgb, "hashtable", aimed_rays(mx, 2000, np.random.default_rng(82), dist=(3.0, 60.0)))
    assert lib.vrm_scene_insert_voxel(s.h, 0, 0, 0, 1) == ERR_STATE     # staging ends with the successful build
