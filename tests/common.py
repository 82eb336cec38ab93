"""Shared helpers for the test-suite (test infrastructure)."""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import pyoracle as po  # noqa: E402
from voxelraymarcher_b200 import scenes  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
COMBOS = [(s, a) for s in ("hashtable", "vcs") for a in ("original", "longestaxis")]

# (origin, look_at, fov) in WORLD units for the probe scene at scale 8; the first is the reference's own (Main.cu:199)
PROBE_CAMERAS = [
    ((6.0, 2.0, 6.0), (0.0, 0.0, -1.0), 60.0),
    ((14.0, 9.0, 12.0), (4.0, 3.0, 2.0), 60.0),
    ((-3.0, 6.0, -9.0), (4.0, 2.0, 2.0), 50.0),
    ((30.0, 20.0, -28.0), (6.0, 3.0, 1.0), 35.0),   # far outside the region table: exercises the scene-entry loop
]

# the mini scene is rendered at scale 1 (camera given directly in voxel units)
MINI_CAMERAS = [((20.0, 18.0, 26.0), (3.0, 2.0, 0.0), 60.0), ((-30.0, 40.0, -35.0), (3.0, 2.0, 4.0), 60.0)]


CONFIG_SAMPLE = 1536    # positions per frame / ray buffer stored in tests/golden/config_golden.npz


def config_sample(n):
    """The fixed, seeded positions (row-major pixels, or rays) of an output of n positions at which tests/golden/config_golden.npz
    stores the configuration tests' results."""
    return np.sort(np.random.default_rng(n).choice(n, CONFIG_SAMPLE, replace=False))


def oracle_kind():
    """The strongest checker available: the unmodified reference built for the host, else its C restatement."""
    return "refh" if po.available("refh") else "orc"


def camera(origin, look_at, fov, width, height, kind=None):
    return po.make_camera(origin, look_at, (0.0, 1.0, 0.0), fov, np.float32(width) / np.float32(height), kind or oracle_kind())


def build_oracle(kind, xyz, rgb, storage):
    s = po.OracleScene(kind)
    s.add_voxels(xyz, rgb)
    s.build(storage)
    return s


def _wide_piece(kind, seed, offset):
    if kind == "terrain":
        xyz, rgb = scenes.terrain(96, seed, max_height=40)
    elif kind == "cube":
        xyz, rgb = scenes.hollow_cube(20, 20, 20, 16)
    else:
        xyz, rgb = scenes.sphere_shell(24, 24, 24, 20, checkered=True)
    return (xyz.astype(np.int64) + np.asarray(offset, np.int64)).astype(np.int32), rgb


# name -> (region range [lo, hi] on every axis, [(piece, seed, voxel offset)]).  Small real content far apart in a table that is mostly
# null regions; two marker voxels at opposite corners force the range (a table always spans region 0, see the header's extent limit).
WIDE_SCENES = {
    "d26": ((0, 25), [("terrain", 11, (700, 0, 900)), ("cube", 0, (40, 1500, 1560)), ("shell", 0, (1580, 1590, 10))]),
    "d200": ((-100, 99), [("terrain", 12, (-5000, -4000, 3000)), ("cube", 0, (4500, 2000, -6000)), ("shell", 0, (-6000, 5000, 5500))]),
    "d512": ((-300, 211), [("terrain", 13, (-19150, -19190, -19130)), ("shell", 0, (13480, 13490, 13470)), ("cube", 0, (-40, 2000, -5000)),
                           ("terrain", 14, (13440, -19190, 6000))]),
    "d1024lo": ((-1023, 0), [("terrain", 15, (-65472, -65472, -65400)), ("cube", 0, (-30, -50, -40)), ("shell", 0, (-40000, -20000, -65470))]),
    "d1024hi": ((0, 1023), [("terrain", 16, (65439, 65400, 65430)), ("cube", 0, (30, 50, 40)), ("shell", 0, (40000, 20000, 65480))]),
}


def wide_scene(name):
    """(xyz, rgb, pieces) of a WIDE_SCENES entry; pieces = [(xyz, rgb)] of its content, the markers not included.  Deterministic."""
    (lo, hi), spec = WIDE_SCENES[name]
    pieces = [_wide_piece(k, seed, off) for k, seed, off in spec]
    markers = np.array([[64 * lo, 64 * lo + 1, 64 * lo + 2], [64 * hi + 63, 64 * hi + 62, 64 * hi + 61]], np.int32)
    xyz = np.concatenate([p[0] for p in pieces] + [markers])
    rgb = np.concatenate([p[1] for p in pieces] + [np.array([0x102030, 0x405060], np.uint32)])
    assert (np.floor_divide(xyz, 64).min(), np.floor_divide(xyz, 64).max()) == (lo, hi), name
    return xyz, rgb, pieces


def horizon_grid(direction, D):
    """vrm_core.cuh horizon_setup restated in float64: (cell width in voxels, nu, nv), or None when the light gets no map."""
    d = np.asarray(direction, np.float32).astype(np.float64)
    n = d / np.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])
    if ((n != 0) & (np.abs(n) < 0.0625)).any():
        return None
    a = np.zeros(3)
    a[int(np.argmin(np.abs(n)))] = 1.0       # least aligned axis (first of equals, as the nested comparisons pick it)
    e1 = np.cross(n, a)
    e1 /= np.linalg.norm(e1)
    e2 = np.cross(n, e1)
    corners = 64.0 * D * np.array([[(c >> i) & 1 for i in range(3)] for c in range(8)], np.float64)
    pad = 4 * np.sqrt(3) + 5.0 + 2.0
    u, v = corners @ e1, corners @ e2
    su, sv = u.max() - u.min() + 2 * pad, v.max() - v.min() + 2 * pad
    cell = 8.0
    while su / cell >= 2048 or sv / cell >= 2048:
        cell *= 2.0
    return cell, int(su / cell) + 1, int(sv / cell) + 1


def lookup_queries(xyz, n_random=20000, seed=1, span=None):
    """Every inserted voxel plus random coordinates (mostly misses) around the scene."""
    rng = np.random.default_rng(seed)
    lo, hi = xyz.min(0) - 70, xyz.max(0) + 70
    if span is not None:
        lo, hi = span
    rnd = rng.integers(lo, hi, size=(n_random, 3)).astype(np.int32)
    return np.ascontiguousarray(np.concatenate([xyz, rnd]).astype(np.int32))
