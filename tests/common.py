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


def lookup_queries(xyz, n_random=20000, seed=1, span=None):
    """Every inserted voxel plus random coordinates (mostly misses) around the scene."""
    rng = np.random.default_rng(seed)
    lo, hi = xyz.min(0) - 70, xyz.max(0) + 70
    if span is not None:
        lo, hi = span
    rnd = rng.integers(lo, hi, size=(n_random, 3)).astype(np.int32)
    return np.ascontiguousarray(np.concatenate([xyz, rnd]).astype(np.int32))
