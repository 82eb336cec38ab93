"""The host build of the shadow horizon map (tests/hostsim/horizon_sim.cpp: hostsim.cpp plus the map's entry points), compiled on first use
into the temporary directory with the flags of tests/hostsim/Makefile -- the repository tree may be read-only -- and cached there by the
hash of its sources.  Used by tests/test_shadow_horizon.py and tools/warp_profile.py."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOSTSIM = os.path.join(ROOT, "tests", "hostsim")
CSRC = os.path.join(ROOT, "voxelraymarcher_b200", "csrc")
SOURCES = [os.path.join(HOSTSIM, "horizon_sim.cpp"), os.path.join(HOSTSIM, "hostsim.cpp")] + \
          [os.path.join(CSRC, f) for f in ("vrm_core.cuh", "vrm_flat.cuh", "vrm_lean.cuh")]
ALGORITHM = {"longestaxis": 0, "original": 1}
STORAGE = {"vcs": 0, "hashtable": 1}
_LIB = None


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
        out = os.path.join(tempfile.gettempdir(), f"vrm_horizon_sim_{h.hexdigest()[:16]}.so")
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


def _f3(v):
    return np.ascontiguousarray(v, np.float32)


def set_lighting(direction, colour=(1.0, 1.0, 1.0), position=(10.0, 10.0, -10.0), use_point=False, use_shadows=True):
    """`direction` as the shadow rays use it (the callers pass the oracle's unit vector, so both sides hold the same floats)."""
    load().sim_set_lighting(_p(_f3(direction)), _p(_f3(colour)), _p(_f3(position)), int(use_point), int(use_shadows))


def set_form(form):
    """hostsim.cpp sim_set_flat: 0 nested, 1 generic state machine, 2 lean machine, 3 state machine with its fast paths per ray."""
    load().sim_set_flat(int(form))


def camera(origin, look_at, fov, aspect):
    out = np.zeros(15, np.float32)
    load().hz_camera_make(_p(_f3(origin)), _p(_f3(look_at)), _p(_f3((0.0, 1.0, 0.0))), C.c_float(fov), C.c_float(aspect), _p(out))
    return out


class Scene:
    def __init__(self, xyz, rgb, storage="vcs", fast=False):
        self.lib = load()
        self.h = C.c_void_p(self.lib.sim_scene_create())
        xyz = np.ascontiguousarray(xyz, np.int32)
        rgb = np.ascontiguousarray(rgb, np.uint32)
        self.lib.sim_scene_add_voxels(self.h, _p(xyz), _p(rgb), C.c_uint64(len(rgb)))
        rc = self.lib.sim_scene_build_vcs_fast(self.h) if fast else self.lib.sim_scene_build(self.h, STORAGE[storage])
        assert rc == 0, rc

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.sim_scene_destroy(self.h)
            self.h = None

    def render(self, cam, w, h, algorithm, scale=1, horizon=True, threads=None, translation=(0.0, 0.0, 0.0)):
        rgb = np.zeros((h, w, 3), np.uint8)
        hits = np.zeros((h, w, 4), np.int32)
        counters = np.zeros(5, np.uint64)
        rc = self.lib.hz_render(self.h, _p(np.ascontiguousarray(cam, np.float32)), _p(_f3(translation)), scale, ALGORITHM[algorithm], w, h,
                                _p(rgb), _p(hits), _p(counters), threads or (os.cpu_count() or 1), int(horizon))
        assert rc == 0, rc
        return dict(rgb=rgb, hits=hits, counters=counters)

    def warp_passes(self, cam, w, h, stride, horizon, threads=None):
        """(tiles, passes, shadow-ray passes) of the lockstep warp simulation of the fused kernel (VCS + longest axis)."""
        out = np.zeros(3, np.uint64)
        rc = self.lib.hz_warp_passes(self.h, _p(np.ascontiguousarray(cam, np.float32)), _p(_f3((0, 0, 0))), 1, w, h, stride, int(horizon),
                                     _p(out), threads or (os.cpu_count() or 1))
        assert rc == 0, rc
        return tuple(int(v) for v in out)

    def property(self, rays, algorithm):
        """hz_property: (shadow rays, violations, rays past their threshold, occupied-cluster tests); None when the light gets no map."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 6)
        out = np.zeros(4, np.uint64)
        rc = self.lib.hz_property(self.h, _p(rays), C.c_uint64(len(rays)), ALGORITHM[algorithm], _p(out))
        if rc == 1:
            return None
        assert rc == 0, rc
        return tuple(int(v) for v in out)
