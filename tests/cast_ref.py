"""The exact ray cast (include/vrm_b200.h "exact ray casts") twice, for the tests of vrm_cast_*:

* ``cast_rays`` / ``cast_views``: a numpy fp32 walk, cell by cell and vectorised over rays, that follows the definition literally -- start
  cell by bisection on tau, then every plane crossing in turn, no leaps.  An origin outside the region table's box may skip to the box
  entry with the per-axis rule (``skip_far``); without it the start cell is searched within ``margin`` cells of the box and the walk steps
  through empty space to the box like any other.
* ``Sim``: the host build of the product's own function (tests/hostsim/cast_sim.cpp around csrc/vrm_core.cuh cast_ray, with leaps),
  compiled on first use into the temporary directory -- the repository tree may be read-only -- and cached there by the hash of its sources.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from tests import surface_ref as sr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOSTSIM = os.path.join(ROOT, "tests", "hostsim")
CSRC = os.path.join(ROOT, "voxelraymarcher_b200", "csrc")
SOURCES = [os.path.join(HOSTSIM, "cast_sim.cpp"), os.path.join(HOSTSIM, "hostsim.cpp")] + \
          [os.path.join(CSRC, f) for f in ("vrm_core.cuh", "vrm_flat.cuh", "vrm_lean.cuh")]
STORAGE = {"vcs": 0, "hashtable": 1}
F32 = np.float32
EMPTY = 1 << 30
_LIB = None


class Stored:
    """The stored voxels of a scene after last-insert-wins, and the region table's box [L, H)^3 (it always contains region 0)."""

    def __init__(self, xyz, rgb):
        xyz = np.asarray(xyz, np.int64).reshape(-1, 3)
        rgb = np.asarray(rgb, np.uint32).reshape(-1)
        reg = np.floor_divide(xyz, 64)
        self.L = 64 * min(0, int(reg.min()))
        self.H = 64 * (max(0, int(reg.max())) + 1)
        self.W = self.H - self.L
        keys, idx = np.unique(self._key(xyz)[::-1], return_index=True)
        self.keys, self.colours = keys, rgb[::-1][idx]

    def _key(self, c):
        c = c - self.L
        return (c[:, 0] * self.W + c[:, 1]) * self.W + c[:, 2]

    def inside(self, c):
        return ((c >= self.L) & (c < self.H)).all(1)

    def lookup(self, c):
        """(found, colour) of integer cells c (n, 3)."""
        c = np.asarray(c, np.int64).reshape(-1, 3)
        ins = self.inside(c)
        key = self._key(np.where(ins[:, None], c, self.L))
        pos = np.minimum(np.searchsorted(self.keys, key), len(self.keys) - 1)
        found = ins & (self.keys[pos] == key)
        return found, np.where(found, self.colours[pos], np.uint32(EMPTY)).astype(np.uint32)


def tau(k, s, d):
    """The definition's plane crossing: ((float)k - s) / d in fp32."""
    with np.errstate(all="ignore"):
        return ((np.asarray(k, np.int64).astype(F32) - s) / d).astype(F32)


def _last_true(pred, lo, hi):
    """Largest k in [lo, hi] with pred(k) for a predicate true up to some k (lo - 1 when none), elementwise."""
    a, b = lo - 1, hi.copy()
    while (a < b).any():
        act = a < b
        m = a + (b - a + 1) // 2
        p = pred(m)
        a = np.where(act & p, m, a)
        b = np.where(act & ~p, m - 1, b)
    return a


def _first_true(pred, lo, hi):
    """Smallest k in [lo, hi] with pred(k) for a predicate true from some k on (hi + 1 when none), elementwise."""
    a, b = lo.copy(), hi + 1
    while (a < b).any():
        act = a < b
        m = (a + b) // 2
        p = pred(m)
        b = np.where(act & p, m, b)
        a = np.where(act & ~p, m + 1, a)
    return a


def cell_after(s, d, X, strict, lo, hi):
    """The cell of one axis (d != 0) after every crossing with tau <= X (strict: < X), searched in [lo, hi] (lo - 1 / hi + 1: beyond)."""
    with np.errstate(invalid="ignore"):
        le = (lambda t: t < X) if strict else (lambda t: t <= X)
        pos = _last_true(lambda k: le(tau(k, s, d)), lo, hi)         # d > 0: max{k : tau(k) <= X}
        neg = _first_true(lambda k: le(tau(k + 1, s, d)), lo, hi)    # d < 0: min{k : tau(k + 1) <= X}
    return np.where(d > 0, pos, neg)


def _walk(st: Stored, P, D, tnear, tfar, scale, translation, skip_far, margin):
    """(hits (n, 4), tau of entry (n,), face (n,), colour (n,), start hit (n,)) of the definition's walk."""
    n = len(P)
    sc = F32(scale)
    with np.errstate(all="ignore"):
        s = (sc * (P - np.asarray(translation, F32))).astype(F32)
        tau0 = (tnear * sc).astype(F32)
        tau1 = (tfar * sc).astype(F32)
    fin = lambda a: np.isfinite(a).all(1) if a.ndim == 2 else np.isfinite(a)  # noqa: E731
    live = fin(P) & fin(D) & fin(tnear) & ~np.isnan(tfar) & ~(tnear > tfar) & fin(s) & fin(tau0)
    L, H = st.L, st.H
    lo = np.full(n, L - 1 if skip_far else L - 1 - margin, np.int64)
    hi = np.full(n, H if skip_far else H + margin, np.int64)
    c = np.zeros((n, 3), np.int64)
    for a in range(3):
        with np.errstate(invalid="ignore"):
            fl = np.floor(s[:, a]).astype(np.float64)
            fl = np.where(np.isfinite(fl), fl, 0.0)
        c[:, a] = np.where(D[:, a] == 0, np.clip(fl, -2.0 ** 40, 2.0 ** 40).astype(np.int64),
                           cell_after(s[:, a], np.where(D[:, a] == 0, F32(1), D[:, a]), tau0, False, lo, hi))
    t = tau0.copy()
    face = np.zeros(n, np.uint8)
    if skip_far:
        # the per-axis rule: enter the box at the latest per-axis entry crossing (ties: the later axis), the other axes by cell_after
        out = live & ~st.inside(c)
        E = np.full(n, -np.inf, F32)
        m = np.full(n, -1, np.int64)
        for a in range(3):
            d = D[:, a]
            below, above = c[:, a] < L, c[:, a] >= H
            away = (below & (d <= 0)) | (above & (d >= 0))
            live &= ~(out & away)
            ent = out & (below | above) & (d != 0)
            Ea = tau(np.where(below, L, H), s[:, a], d)
            take = ent & ((m < 0) | (Ea >= E))
            E = np.where(take, Ea, E)
            m = np.where(take, a, m)
        go = out & live & (E <= tau1)
        live &= ~(out & ~go)
        newc = c.copy()
        for b in range(3):
            d = D[:, b]
            cb = cell_after(s[:, b], np.where(d == 0, F32(1), d), E, False, np.full(n, L - 1), np.full(n, H))
            cbs = cell_after(s[:, b], np.where(d == 0, F32(1), d), E, True, np.full(n, L - 1), np.full(n, H))
            newc[:, b] = np.where(m == b, np.where(d > 0, L, H - 1), np.where(d == 0, c[:, b], np.where(b > m, cbs, cb)))
        c = np.where(go[:, None], newc, c)
        live &= ~(go & ~st.inside(c))
        t = np.where(go, E, t)
        face = np.where(go, 1 + 2 * m + (np.take_along_axis(D, np.maximum(m, 0)[:, None], 1)[:, 0] < 0), face).astype(np.uint8)
    hits = np.zeros((n, 4), np.int32)
    tau_hit = np.zeros(n, F32)
    face_hit = np.zeros(n, np.uint8)
    colour = np.full(n, EMPTY, np.uint32)
    idx = np.nonzero(live)[0]
    c, t, face = c[idx], t[idx], face[idx]
    while len(idx):
        # a cell outside the box with an axis that can never come back: the walk finds nothing more
        never = np.zeros(len(idx), bool)
        for a in range(3):
            d = D[idx, a]
            never |= ((c[:, a] < L) & (d <= 0)) | ((c[:, a] >= H) & (d >= 0))
        found, col = st.lookup(c)
        done = found | never
        if found.any():
            j = idx[found]
            hits[j, :3] = c[found]
            hits[j, 3] = 1
            tau_hit[j], face_hit[j], colour[j] = t[found], face[found], col[found]
        keep = ~done
        idx, c, t, face = idx[keep], c[keep], t[keep], face[keep]
        if not len(idx):
            break
        # the next crossing: the smallest, ties to the earlier axis
        best = np.zeros(len(idx), F32)
        m = np.full(len(idx), -1, np.int64)
        for a in range(3):
            d = D[idx, a]
            nta = tau(np.where(d > 0, c[:, a] + 1, c[:, a]), s[idx, a], d)
            take = (d != 0) & ((m < 0) | (nta < best))
            best = np.where(take, nta, best)
            m = np.where(take, a, m)
        go = (m >= 0) & (best <= tau1[idx])
        idx, c, t, face, best, m = idx[go], c[go], t[go], face[go], best[go], m[go]
        dm = np.take_along_axis(D[idx], m[:, None], 1)[:, 0]
        c[np.arange(len(idx)), m] += np.where(dm > 0, 1, -1)
        t = best
        face = (1 + 2 * m + (dm < 0)).astype(np.uint8)
    return hits, tau_hit, face_hit, colour


def cast_rays(st: Stored, rays, ranges=None, scale=1, translation=(0.0, 0.0, 0.0), skip_far=True, margin=6000):
    """dict(hits (n, 4) int32, depth (n,) float32, face (n,) uint8, colour (n,) uint32) of world rays (n, 6), ranges (n, 2) or None."""
    r = np.asarray(rays, F32).reshape(-1, 6)
    n = len(r)
    rg = np.tile(np.array([0.0, np.inf], F32), (n, 1)) if ranges is None else np.asarray(ranges, F32).reshape(-1, 2)
    hits, t, face, colour = _walk(st, r[:, :3], r[:, 3:], rg[:, 0], rg[:, 1], scale, translation, skip_far, margin)
    with np.errstate(all="ignore"):
        depth = np.where(face == 0, rg[:, 0], t / F32(scale)).astype(F32)
    depth = np.where(hits[:, 3] != 0, depth, F32(np.inf)).astype(F32)
    return dict(hits=hits, depth=depth, face=face, colour=colour)


def cast_pixels(st: Stored, cam, width, height, pixels, scale=1, translation=(0.0, 0.0, 0.0)):
    """``cast_views`` of one camera at the row-major pixel indices ``pixels`` only: dict of (m, ...) arrays."""
    P, D, length = sr.pixel_rays(cam, width, height)
    P, D, length = P.reshape(-1, 3)[pixels], D.reshape(-1, 3)[pixels], length.reshape(-1)[pixels]
    n = len(P)
    hits, t, face, colour = _walk(st, P, D, np.zeros(n, F32), np.full(n, np.inf, F32), scale, translation, True, 0)
    with np.errstate(all="ignore"):
        depth = np.where(face == 0, length, (length + t / F32(scale)).astype(F32)).astype(F32)
    return dict(hits=hits, depth=np.where(hits[:, 3] != 0, depth, F32(np.inf)).astype(F32), face=face, colour=colour)


def cast_views(st: Stored, cameras, width, height, scale=1, translation=(0.0, 0.0, 0.0)):
    """The same per pixel of each camera's frame (primary_ray's rays over [0, +inf)), view-major: (n, H, W[, 4])."""
    out = {k: [] for k in ("hits", "depth", "face", "colour")}
    for cam in cameras:
        P, D, length = sr.pixel_rays(cam, width, height)
        P, D, length = P.reshape(-1, 3), D.reshape(-1, 3), length.reshape(-1)
        n = len(P)
        hits, t, face, colour = _walk(st, P, D, np.zeros(n, F32), np.full(n, np.inf, F32), scale, translation, True, 0)
        with np.errstate(all="ignore"):
            depth = np.where(face == 0, length, (length + t / F32(scale)).astype(F32)).astype(F32)
        depth = np.where(hits[:, 3] != 0, depth, F32(np.inf)).astype(F32)
        for k, v in (("hits", hits.reshape(height, width, 4)), ("depth", depth.reshape(height, width)),
                     ("face", face.reshape(height, width)), ("colour", colour.reshape(height, width))):
            out[k].append(v)
    return {k: np.stack(v) for k, v in out.items()}


def same(a, b):
    """Bit-identical cast results."""
    return all(np.array_equal(a[k], b[k]) for k in ("hits", "face", "colour")) and sr.same_bits(a["depth"], b["depth"])


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
        out = os.path.join(tempfile.gettempdir(), f"vrm_cast_sim_{h.hexdigest()[:16]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            cmd = ["g++", "-std=c++17", "-O2", "-ffp-contract=off"] + (["-mfma"] if _has_fma() else []) + \
                  ["-fPIC", "-shared", "-fopenmp", SOURCES[0], "-o", tmp]
            subprocess.run(cmd, check=True)
            os.replace(tmp, out)
        _LIB = C.CDLL(out)
        _LIB.sim_scene_create.restype = C.c_void_p
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Sim:
    """A scene built by the host harness, cast by the product's cast_ray."""

    def __init__(self, xyz, rgb, storage):
        self.lib = load()
        self.h = C.c_void_p(self.lib.sim_scene_create())
        xyz = np.ascontiguousarray(xyz, np.int32)
        rgb = np.ascontiguousarray(rgb, np.uint32)
        self.lib.sim_scene_add_voxels(self.h, _p(xyz), _p(rgb), C.c_uint64(len(rgb)))
        assert self.lib.sim_scene_build(self.h, STORAGE[storage]) == 0

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.sim_scene_destroy(self.h)
            self.h = None

    def lookup(self, xyz):
        xyz = np.ascontiguousarray(xyz, np.int32).reshape(-1, 3)
        out = np.zeros(len(xyz), np.uint32)
        assert self.lib.sim_lookup(self.h, _p(xyz), C.c_uint64(len(xyz)), _p(out), None) == 0
        return out

    def cast_rays(self, rays, ranges=None, scale=1, translation=(0.0, 0.0, 0.0)):
        r = np.ascontiguousarray(rays, F32).reshape(-1, 6)
        n = len(r)
        rg = None if ranges is None else np.ascontiguousarray(ranges, F32).reshape(-1, 2)
        out = dict(hits=np.zeros((n, 4), np.int32), depth=np.zeros(n, F32), face=np.zeros(n, np.uint8), colour=np.zeros(n, np.uint32))
        assert self.lib.cast_rays(self.h, _p(r), None if rg is None else _p(rg), C.c_uint64(n), _p(np.ascontiguousarray(translation, F32)),
                                  C.c_uint32(scale), _p(out["hits"]), _p(out["depth"]), _p(out["face"]), _p(out["colour"])) == 0
        return out

    def cast_views(self, cameras, width, height, scale=1, translation=(0.0, 0.0, 0.0)):
        cams = np.ascontiguousarray(np.stack([np.asarray(c, F32) for c in cameras]), F32)
        v = len(cams)
        out = dict(hits=np.zeros((v, height, width, 4), np.int32), depth=np.zeros((v, height, width), F32),
                   face=np.zeros((v, height, width), np.uint8), colour=np.zeros((v, height, width), np.uint32))
        assert self.lib.cast_views(self.h, _p(cams), C.c_uint32(v), _p(np.ascontiguousarray(translation, F32)), C.c_uint32(scale),
                                   C.c_uint32(width), C.c_uint32(height), _p(out["hits"]), _p(out["depth"]), _p(out["face"]), _p(out["colour"])) == 0
        return out


# ---- test inputs shared by tests/test_cast.py (host build) and tests/test_cast_gpu.py (kernel) ------------------------------------------
TIE_DIRS = np.array([(1, 1, 0), (1, 1, 1), (2, 1, 0), (1, -1, 1)], np.float32)


def _world(s, scale, translation):
    return (np.asarray(s, np.float64) / scale + np.asarray(translation, np.float64)).astype(F32)


def ray_cases(st: Stored, scale=1, translation=(0.0, 0.0, 0.0), seed=0, n=1500):
    """dict name -> world rays (m, 6) for the scene `st`, built in the local frame and converted with P = s / scale + translation."""
    rng = np.random.default_rng(seed)
    L, H = st.L, st.H
    vox = np.stack([st.keys // (st.W * st.W), (st.keys // st.W) % st.W, st.keys % st.W], 1) + L
    pick = lambda m: vox[rng.integers(0, len(vox), m)].astype(np.float64)  # noqa: E731
    out = {}

    def zeroed(d):
        m = len(d)
        k = rng.integers(0, 8, m)
        ax = rng.integers(0, 3, m)
        d[k == 1, ax[k == 1]] = 0.0
        d[k == 2, ax[k == 2]] = -0.0
        for i in np.nonzero(k == 3)[0]:
            d[i, [a for a in range(3) if a != ax[i]]] = 0.0           # axis-aligned
        return d

    # random origins around the box, towards stored voxels or anywhere
    org = rng.uniform(L - 40, H + 40, (n, 3))
    tgt = pick(n) + rng.uniform(0, 1, (n, 3))
    d = np.where(rng.random((n, 1)) < 0.7, tgt - org, rng.normal(size=(n, 3)))
    out["random"] = (org, zeroed(d.astype(F32)))
    # exact ties: integer / half-integer origins on diagonals through cluster and region corners
    corner = pick(n)
    corner = np.where(rng.random((n, 1)) < 0.5, np.floor(corner / 8) * 8, np.floor(corner / 64) * 64)
    d = TIE_DIRS[rng.integers(0, 4, n)][:, rng.permutation(3)] * np.where(rng.random((n, 3)) < 0.5, -1, 1)
    d = np.stack([dd[rng.permutation(3)] for dd in d])
    org = corner - rng.integers(1, 40, (n, 1)) * d + np.where(rng.random((n, 1)) < 0.3, 0.5, 0.0)
    out["ties"] = (org, d.astype(F32))
    # origins on cluster / region planes, and inside stored voxels
    org = pick(n) + rng.uniform(0, 1, (n, 3))
    snap = rng.integers(0, 3, n)
    step = np.where(rng.random(n) < 0.5, 8, 64)
    org[np.arange(n), snap] = np.round(org[np.arange(n), snap] / step) * step
    d = pick(n) + 0.5 - org
    out["planes"] = (org, zeroed(d.astype(F32)))
    org = pick(n) + np.where(rng.random((n, 1)) < 0.3, 0.0, rng.uniform(0, 1, (n, 3)))
    out["inside"] = (org, zeroed(rng.normal(size=(n, 3)).astype(F32)))
    # far outside the box (up to a few thousand cells), hitting or missing it
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    tgt = pick(n) + 0.5
    org = tgt + u * rng.uniform(H - L, H - L + 3000, (n, 1))
    d = tgt - org + np.where(rng.random((n, 1)) < 0.3, rng.normal(0, H - L, (n, 3)), 0.0)
    out["far"] = (org, d.astype(F32))
    # |s| so large that tau_a has runs of equal values
    org = tgt + u * rng.uniform(2.0 ** 24, 2.0 ** 26, (n, 1))
    out["runs"] = (org, (tgt - org).astype(F32))
    return {k: np.concatenate([_world(o, scale, translation), dd.astype(F32)], 1) for k, (o, dd) in out.items()}


def moderate_rays(st: Stored, scale=1, translation=(0.0, 0.0, 0.0), seed=1, n=1500):
    """Origins 1..300 cells outside the box, for checking the skip to the box entry against plain stepping."""
    rng = np.random.default_rng(seed)
    vox = np.stack([st.keys // (st.W * st.W), (st.keys // st.W) % st.W, st.keys % st.W], 1) + st.L
    tgt = vox[rng.integers(0, len(vox), n)] + 0.5
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    centre = (st.L + st.H) / 2.0
    org = centre + u * ((st.H - st.L) * 0.87 + rng.uniform(1, 300, (n, 1)))
    d = tgt - org + rng.normal(0, 8, (n, 3))
    return np.concatenate([_world(org, scale, translation), d.astype(F32)], 1)


def range_cases(n, seed=2):
    """dict name -> ranges (n, 2) {t_near, t_far} in world units (None: [0, +inf))."""
    rng = np.random.default_rng(seed)
    a = rng.uniform(-10, 60, n).astype(F32)
    b = (a + rng.uniform(0, 120, n)).astype(F32)
    out = {"default": None, "interval": np.stack([a, b], 1)}
    out["negative_near"] = np.stack([-np.abs(a), b], 1)
    out["point"] = np.stack([a, a], 1)
    out["reversed"] = np.stack([b + 1, a], 1)
    special = np.stack([a, b], 1)
    k = rng.integers(0, 6, n)
    special[k == 0, 0] = np.nan
    special[k == 1, 1] = np.nan
    special[k == 2, 1] = np.inf
    special[k == 3, 0] = np.inf
    special[k == 4, 0] = -np.inf
    out["special"] = special
    return {k: (None if v is None else np.ascontiguousarray(v, F32)) for k, v in out.items()}
