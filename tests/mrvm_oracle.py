"""ctypes binding of the MultiResolutionVoxelMap oracle (tests/cpp/mrvm_oracle.cc): a serial one-thread restatement
of builder/multi_resolution_voxel_map.cc, the parity checker of the sm_mrvm_* entry points.  TEST INFRASTRUCTURE:
only tests/ and profiles/time_mrvm.py import this module.

The library is compiled with g++ on first use into a directory under the system temporary directory, named after a
hash of the source and flags, so the repository tree is never written to."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpp", "mrvm_oracle.cc")
# the flags of the other oracle pieces (oracle/Makefile): no FMA contraction, so float sums keep their order
_FLAGS = ["-O2", "-fPIC", "-std=c++17", "-ffp-contract=off", "-Wall", "-Wextra", "-shared"]
_lib = None


def _build():
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if cxx is None:
        raise RuntimeError("g++ is needed to build the MultiResolutionVoxelMap oracle")
    with open(_SRC, "rb") as f:
        tag = hashlib.sha1(f.read() + " ".join(_FLAGS).encode()).hexdigest()[:16]
    d = os.path.join(tempfile.gettempdir(), f"sm_mrvm_oracle_{os.getuid()}_{tag}")
    so = os.path.join(d, "libmrvm_oracle.so")
    if not os.path.exists(so):
        os.makedirs(d, exist_ok=True)
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=d)
        os.close(fd)
        subprocess.check_call([cxx, *_FLAGS, "-o", tmp, _SRC])
        os.replace(tmp, so)                      # atomic: concurrent test processes see a whole library or none
    return so
class MrvmSettings(C.Structure):
    _fields_ = [("output_average", C.c_int32), ("output_rgb", C.c_int32), ("use_max_intensity", C.c_int32),
                ("prob_threshold", C.c_float), ("low_resolution", C.c_float), ("high_resolution", C.c_float),
                ("hit_prob", C.c_float), ("miss_prob", C.c_float), ("z_offset", C.c_float),
                ("max_point_num_in_cell", C.c_int32)]


def mrvm_settings(**kw):
    """MrvmSettings with the reference's defaults (multi_resolution_voxel_map.h:55-66), overridden by kw."""
    s = MrvmSettings(0, 0, 1, 0.6, 1.0, 0.1, 0.55, 0.48, 0.0, 10)
    for k, v in kw.items():
        setattr(s, k, v)
    return s


def _mrvm_lib():
    global _lib
    if _lib is not None:
        return _lib
    L = C.CDLL(_build())
    vp, i64 = C.c_void_p, C.c_int64
    L.sm_oracle_mrvm_create.restype = vp
    L.sm_oracle_mrvm_create.argtypes = [C.POINTER(MrvmSettings)]
    L.sm_oracle_mrvm_destroy.argtypes = [vp]
    L.sm_oracle_mrvm_set_offset_z.argtypes = [vp, C.c_float]
    L.sm_oracle_mrvm_size.restype = i64
    L.sm_oracle_mrvm_size.argtypes = [vp]
    L.sm_oracle_mrvm_insert.restype = i64
    L.sm_oracle_mrvm_insert.argtypes = [vp, vp, i64, vp]
    L.sm_oracle_mrvm_output.restype = i64
    L.sm_oracle_mrvm_output.argtypes = [vp, C.c_float, C.c_int32, vp, i64]
    L.sm_oracle_mrvm_state.restype = i64
    L.sm_oracle_mrvm_state.argtypes = [vp, vp, vp, vp, vp, vp, i64]
    L.sm_oracle_voxel_casting_bresenham.restype = i64
    L.sm_oracle_voxel_casting_bresenham.argtypes = [vp, vp, C.c_float, vp, i64]
    _lib = L
    return L


class Mrvm:
    """Serial restatement of MultiResolutionVoxelMap (one thread, output in ascending key order)."""

    def __init__(self, **settings):
        self.settings = mrvm_settings(**settings)
        self._L = _mrvm_lib()
        self._h = self._L.sm_oracle_mrvm_create(C.byref(self.settings))
        if not self._h:
            raise ValueError("invalid MrvmSettings")

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.sm_oracle_mrvm_destroy(self._h)
            self._h = None

    def SetOffsetZ(self, z):
        self._L.sm_oracle_mrvm_set_offset_z(self._h, float(z))

    def size(self):
        return self._L.sm_oracle_mrvm_size(self._h)

    def InsertPointCloud(self, points5, origin):
        """-> number of dropped points, -1 out of range (map unchanged), -2 ray-end CHECK failure."""
        p = np.ascontiguousarray(np.asarray(points5, dtype=np.float32))
        assert p.ndim == 2 and p.shape[1] == 5
        o = np.ascontiguousarray(np.asarray(origin, dtype=np.float32).reshape(3))
        return self._L.sm_oracle_mrvm_insert(self._h, p.ctypes.data, p.shape[0], o.ctypes.data)

    def OutputToPointCloud(self, threshold, rgb=False):
        m = self._L.sm_oracle_mrvm_output(self._h, float(threshold), int(rgb), None, 0)
        out = np.zeros((max(m, 1), 4), np.float32)
        got = self._L.sm_oracle_mrvm_output(self._h, float(threshold), int(rgb), out.ctypes.data, m)
        assert got == m
        return out[:m].copy()

    def State(self):
        """dict(keys, prob, max_intensity, npts, points (n, max_point_num_in_cell, 4)) in ascending key order."""
        mp = self.settings.max_point_num_in_cell
        n = self.size()
        keys = np.zeros(n, np.int64); prob = np.zeros(n, np.uint8)
        mi = np.zeros(n, np.int32); npts = np.zeros(n, np.int32); pts = np.zeros((n, mp, 4), np.float32)
        got = self._L.sm_oracle_mrvm_state(self._h, keys.ctypes.data, prob.ctypes.data, mi.ctypes.data, npts.ctypes.data,
                                           pts.ctypes.data, n)
        assert got == n
        return {"keys": keys, "prob": prob, "max_intensity": mi, "npts": npts, "points": pts}


def voxel_casting_bresenham(start, end, step):
    """common::VoxelCastingBresenham -> (n, 3) int32 voxels, or the negative error code."""
    a = np.ascontiguousarray(np.asarray(start, np.float32).reshape(3))
    b = np.ascontiguousarray(np.asarray(end, np.float32).reshape(3))
    L = _mrvm_lib()
    n = L.sm_oracle_voxel_casting_bresenham(a.ctypes.data, b.ctypes.data, float(step), None, 0)
    if n < 0:
        return n
    out = np.zeros((n, 3), np.int32)
    L.sm_oracle_voxel_casting_bresenham(a.ctypes.data, b.ctypes.data, float(step), out.ctypes.data, n)
    return out
