"""The hit-surface definition (include/vrm_b200.h "hit surfaces") twice, for the tests of vrm_hit_surface_*:

* ``views`` / ``rays``: a numpy fp32 restatement, operation by operation (every numpy float32 operation rounds to nearest once);
* ``sim_views`` / ``sim_rays``: the host build of the product's own definition (tests/hostsim/surface_sim.cpp around csrc/vrm_core.cuh
  primary_ray + hit_surface), compiled on first use into the temporary directory -- the repository tree may be read-only -- and cached
  there by the hash of its sources.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCES = [os.path.join(ROOT, "tests", "hostsim", "surface_sim.cpp"), os.path.join(ROOT, "voxelraymarcher_b200", "csrc", "vrm_core.cuh")]
F32 = np.float32
_LIB = None


def pixel_rays(cam, width, height):
    """primary_ray (calculateWorldRay) for every pixel, row 0 = top: P (H, W, 3), D (H, W, 3) and len (H, W), all float32."""
    cam = np.asarray(cam, F32)
    x = np.arange(width, dtype=np.uint32)[None, :]
    y = np.arange(height, dtype=np.uint32)[:, None]
    u = (x.astype(F32) + F32(0.5)) / F32(width)
    v = ((np.uint32(height) - y).astype(F32) + F32(0.5)) / F32(height)
    o = [(cam[3 + i] + u * cam[6 + i]) + v * cam[9 + i] for i in range(3)]
    rel = [o[i] - cam[i] for i in range(3)]
    length = np.sqrt((rel[0] * rel[0] + rel[1] * rel[1]) + rel[2] * rel[2])
    d = [rel[i] / length for i in range(3)]
    return np.stack(o, -1).astype(F32), np.stack(d, -1).astype(F32), length.astype(F32)


def slab(hits, P, D, translation, scale):
    """(t, face) of the definition for records hits (n, 4) and rays P, D (n, 3), before the conversion to depth."""
    hits = np.asarray(hits, np.int32).reshape(-1, 4)
    P = np.asarray(P, F32).reshape(-1, 3)
    D = np.asarray(D, F32).reshape(-1, 3)
    sc = F32(scale)
    t = np.zeros(len(hits), F32)
    face = np.zeros(len(hits), np.uint8)
    with np.errstate(all="ignore"):
        for a in range(3):
            d = D[:, a]
            s = sc * (P[:, a] - F32(translation[a]))
            h = hits[:, a].astype(np.int64)
            f = np.where(d > 0, h, h + 1).astype(F32)
            ta = (f - s) / d
            take = (d != 0) & ((face == 0) | (ta > t))
            t = np.where(take, ta, t).astype(F32)
            face = np.where(take, 1 + 2 * a + (d < 0), face).astype(np.uint8)
    return t, face


def _finish(hits, t, face, scale, length):
    with np.errstate(all="ignore"):
        q = t / F32(scale)
        depth = q if length is None else (length + q)
    depth = np.where(face == 0, F32(np.nan), depth).astype(F32)
    flag = hits.reshape(-1, 4)[:, 3] != 0
    return np.where(flag, depth, F32(np.inf)).astype(F32), np.where(flag, face, 0).astype(np.uint8)


def views(hits, cameras, width, height, scale=1, translation=(0.0, 0.0, 0.0)):
    """depth, face of a view-major hit map (n, H, W, 4) for n cameras, each (n, H, W)."""
    hits = np.asarray(hits, np.int32).reshape(-1, height, width, 4)
    depth, face = [], []
    for v, cam in enumerate(cameras):
        P, D, length = pixel_rays(cam, width, height)
        t, f = slab(hits[v], P, D, translation, scale)
        dv, fv = _finish(hits[v], t, f, scale, length.reshape(-1))
        depth.append(dv.reshape(height, width)); face.append(fv.reshape(height, width))
    return np.stack(depth), np.stack(face)


def rays(hits, ray_array, scale=1, translation=(0.0, 0.0, 0.0)):
    """depth, face of traced rays (n, 6) and their hit records (n, 4), each (n,)."""
    r = np.asarray(ray_array, F32).reshape(-1, 6)
    hits = np.asarray(hits, np.int32).reshape(-1, 4)
    t, f = slab(hits, r[:, :3], r[:, 3:], translation, scale)
    return _finish(hits, t, f, scale, None)


def same_bits(a, b):
    """Bit-identical float32 arrays, any NaN matching any NaN."""
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def entry_distance(hits, P, D, translation, scale):
    """Distance (local voxel units, float64) of the entry point s + t D from the hit voxel's box, per record with flag != 0."""
    hits = np.asarray(hits, np.int32).reshape(-1, 4)
    P = np.asarray(P, F32).reshape(-1, 3)
    D = np.asarray(D, F32).reshape(-1, 3)
    t, _ = slab(hits, P, D, translation, scale)
    keep = hits[:, 3] != 0
    s = (F32(scale) * (P - np.asarray(translation, F32))).astype(np.float64)
    e = s + t.astype(np.float64)[:, None] * D.astype(np.float64)
    lo = hits[:, :3].astype(np.float64)
    out = np.maximum(np.maximum(lo - e, e - (lo + 1.0)), 0.0)
    return np.sqrt((out * out).sum(1))[keep]


def _has_fma():
    try:
        with open("/proc/cpuinfo") as f:
            return " fma" in f.read()
    except OSError:
        return False


def load():
    global _LIB
    if _LIB is None:
        h = hashlib.sha1()
        for p in SOURCES:
            with open(p, "rb") as f:
                h.update(f.read())
        out = os.path.join(tempfile.gettempdir(), f"vrm_surface_sim_{h.hexdigest()[:16]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            cmd = ["g++", "-std=c++17", "-O2", "-ffp-contract=off"] + (["-mfma"] if _has_fma() else []) + ["-fPIC", "-shared", SOURCES[0], "-o", tmp]
            subprocess.run(cmd, check=True)
            os.replace(tmp, out)
        _LIB = C.CDLL(out)
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def sim_views(hits, cameras, width, height, scale=1, translation=(0.0, 0.0, 0.0)):
    cams = np.ascontiguousarray(np.stack([np.asarray(c, F32) for c in cameras]), F32)
    n = cams.shape[0]
    hits = np.ascontiguousarray(hits, np.int32)
    assert hits.size == n * height * width * 4
    depth = np.empty((n, height, width), F32)
    face = np.empty((n, height, width), np.uint8)
    load().surf_views(_p(cams), C.c_uint32(n), _p(np.ascontiguousarray(translation, F32)), C.c_uint32(scale), C.c_uint32(width), C.c_uint32(height),
                      _p(hits), _p(depth), _p(face))
    return depth, face


def sim_rays(hits, ray_array, scale=1, translation=(0.0, 0.0, 0.0)):
    r = np.ascontiguousarray(ray_array, F32).reshape(-1, 6)
    hits = np.ascontiguousarray(hits, np.int32).reshape(-1, 4)
    n = r.shape[0]
    depth = np.empty(n, F32)
    face = np.empty(n, np.uint8)
    load().surf_rays(_p(r), C.c_uint64(n), _p(np.ascontiguousarray(translation, F32)), C.c_uint32(scale), _p(hits), _p(depth), _p(face))
    return depth, face
