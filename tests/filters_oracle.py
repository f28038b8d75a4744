"""ctypes binding of the filter-chain oracle (tests/cpp/filters_oracle.cc): a serial restatement of
pre_processers::filter::Factory and its nine filters, the parity checker of the sm_filter_chain_* entry points.
TEST INFRASTRUCTURE: only tests/ and profiles/time_filters.py import this module.

`Chain` has the methods of staticmapping_b200.FilterChain, so the Python filter classes run on it unchanged
(``smb.Range(chain=Chain())``).  The library is compiled with g++ on first use into a directory under the system
temporary directory, named after a hash of the source and flags, so the repository tree is never written to."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpp", "filters_oracle.cc")
_FLAGS = ["-O2", "-fPIC", "-std=c++17", "-ffp-contract=off", "-Wall", "-Wextra", "-shared"]
_lib = None

ANGLE_HOST = 0      # the host C library's atan2f: the literal reference
ANGLE_PRODUCT = 1   # the engine's angle function


def _build():
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if cxx is None:
        raise RuntimeError("g++ is needed to build the filter-chain oracle")
    with open(_SRC, "rb") as f:
        tag = hashlib.sha1(f.read() + " ".join(_FLAGS).encode()).hexdigest()[:16]
    d = os.path.join(tempfile.gettempdir(), f"sm_filters_oracle_{os.getuid()}_{tag}")
    so = os.path.join(d, "libfilters_oracle.so")
    if not os.path.exists(so):
        os.makedirs(d, exist_ok=True)
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=d)
        os.close(fd)
        subprocess.check_call([cxx, *_FLAGS, "-o", tmp, _SRC])
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is not None:
        return _lib
    L = C.CDLL(_build())
    vp, i64 = C.c_void_p, C.c_int64
    L.sm_oracle_filter_chain_create.restype = vp
    L.sm_oracle_filter_chain_destroy.argtypes = [vp]
    L.sm_oracle_filter_set_angle_mode.argtypes = [C.c_int]
    L.sm_oracle_filter_chain_add.argtypes = [vp, C.c_char_p]
    L.sm_oracle_filter_chain_set_param.argtypes = [vp, C.c_int, C.c_char_p, C.c_int, C.c_char_p]
    L.sm_oracle_filter_chain_valid.argtypes = [vp, C.c_int]
    L.sm_oracle_filter_chain_set_seed.argtypes = [vp, C.c_uint64]
    L.sm_oracle_filter_chain_filter.restype = i64
    L.sm_oracle_filter_chain_filter.argtypes = [vp, vp, i64, vp, vp]
    L.sm_oracle_filter_chain_stage_counts.argtypes = [vp, vp, C.c_int]
    L.sm_oracle_gr2_state.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp, vp]
    _lib = L
    return L


def set_angle_mode(mode):
    lib().sm_oracle_filter_set_angle_mode(int(mode))


class Chain:
    """Serial Factory with the interface of staticmapping_b200.FilterChain."""

    def __init__(self, angle_mode=ANGLE_PRODUCT):
        self.angle_mode = angle_mode
        self._L = lib()
        self._h = self._L.sm_oracle_filter_chain_create()

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.sm_oracle_filter_chain_destroy(self._h)
            self._h = None

    def add(self, name):
        return self._L.sm_oracle_filter_chain_add(self._h, name.encode())

    def set_param(self, stage, name, type_, text):
        return self._L.sm_oracle_filter_chain_set_param(self._h, stage, name.encode(), type_, text.encode())

    def valid(self, stage):
        return self._L.sm_oracle_filter_chain_valid(self._h, stage)

    def set_seed(self, seed):
        self._L.sm_oracle_filter_chain_set_seed(self._h, int(seed) & ((1 << 64) - 1))
        return 0

    def filter(self, points5):
        p = np.ascontiguousarray(points5, np.float32)
        n = p.shape[0]
        out = np.empty((max(n, 1), 5), np.float32)
        kept = np.empty(max(n, 1), np.int32)
        set_angle_mode(self.angle_mode)
        m = self._L.sm_oracle_filter_chain_filter(self._h, p.ctypes.data, n, out.ctypes.data, kept.ctypes.data)
        if m < 0:
            return -1, out[:0].copy(), kept[:0].copy()
        return 0, out[:m].copy(), kept[:m].copy()

    def stage_counts(self):
        ns = self._L.sm_oracle_filter_chain_stage_counts(self._h, None, 0)
        c = np.zeros(max(ns, 1), np.int64)
        self._L.sm_oracle_filter_chain_stage_counts(self._h, c.ctypes.data, ns)
        return c[:ns]


GR2_DEFAULTS = dict(r_max=100.0, r_min=1.0, start_ground_height=-0.25, long_line_threshold=1.0,
                    max_long_line_height=0.1, max_start_height=0.2, max_error=0.05,
                    max_slope=float(np.float32(np.tan(np.pi / 12))), max_b=0.1, max_dist_to_line=0.05,
                    search_angle=10.0, bin_num=200, segment_num=180)
GR2_ORDER = ["r_max", "r_min", "start_ground_height", "long_line_threshold", "max_long_line_height",
             "max_start_height", "max_error", "max_slope", "max_b", "max_dist_to_line", "search_angle", "bin_num",
             "segment_num"]


def gr2_state(points5, angle_mode=ANGLE_PRODUCT, **kw):
    """GroundRemoval2's binning and FitLines -> dict(cell, member, cell_dz, cell_used, lines (S, cap, 4), nlines)."""
    P = dict(GR2_DEFAULTS, **kw)
    params = np.array([P[k] for k in GR2_ORDER], np.float32)
    p = np.ascontiguousarray(points5, np.float32)
    n = p.shape[0]
    B, S = int(P["bin_num"]), int(P["segment_num"])
    cap = B // 2 + 2
    cell = np.zeros(n, np.int32); member = np.zeros(n, np.uint8)
    cell_dz = np.zeros((S * B, 2), np.float32); cell_used = np.zeros(S * B, np.uint8)
    lines = np.zeros((S, cap, 4), np.float32); nlines = np.zeros(S, np.int32)
    set_angle_mode(angle_mode)
    lib().sm_oracle_gr2_state(p.ctypes.data, n, params.ctypes.data, cell.ctypes.data, member.ctypes.data,
                              cell_dz.ctypes.data, cell_used.ctypes.data, lines.ctypes.data, nlines.ctypes.data)
    return dict(cell=cell, member=member, cell_dz=cell_dz, cell_used=cell_used, lines=lines, nlines=nlines)


def run_chain(stages, points5, seed=0, angle_mode=ANGLE_PRODUCT, calls=1):
    """stages: [(name, {param: (type, text)})] -> (rc, out, kept) of the last of `calls` Filter calls."""
    c = Chain(angle_mode)
    c.set_seed(seed)
    for name, params in stages:
        k = c.add(name)
        assert k >= 0, name
        for pname, (t, text) in params.items():
            assert c.set_param(k, pname, t, text) == 0, pname
    r = None
    for _ in range(calls):
        r = c.filter(points5)
    return r
