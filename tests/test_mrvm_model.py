"""MultiResolutionVoxelMap without a GPU: the serial oracle on hand-computed cases, a numpy model of the counting
formulation the kernels use (misses before hits, binary lifting) against the oracle bit for bit over multi-scan
scenes, and the product's __host__ __device__ Bresenham walk and voxel update through the host hooks."""
import ctypes as C

import numpy as np
import pytest

import mrvm_oracle as O
from staticmapping_b200 import _lib

HALF = 1 << 20


def pts5(xyz, intensity=None):
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    p = np.zeros((xyz.shape[0], 5), np.float32)
    p[:, :3] = xyz
    p[:, 3] = 0 if intensity is None else intensity
    return p


def key(ix, iy, iz):
    return ((ix + HALF) << 42) | ((iy + HALF) << 21) | (iz + HALF)


def one_step_tables(hit=0.55, miss=0.48):
    """the product's one-step hit / miss maps (test hook sm_debug_mrvm_update)"""
    tab = np.zeros(512, np.uint8)
    z = np.zeros(0, np.int64)
    assert _lib.lib().sm_debug_mrvm_update(hit, miss, None, z.ctypes.data, z.ctypes.data, 0, None, tab.ctypes.data) == 0
    return tab[:256].copy(), tab[256:].copy()


def hook_update(probs, misses, hits, hit=0.55, miss=0.48):
    p = np.ascontiguousarray(probs, np.uint8)
    m = np.ascontiguousarray(misses, np.int64); h = np.ascontiguousarray(hits, np.int64)
    out = np.zeros_like(p)
    rc = _lib.lib().sm_debug_mrvm_update(hit, miss, p.ctypes.data, m.ctypes.data, h.ctypes.data, p.size, out.ctypes.data,
                                         None)
    assert rc == 0
    return out


def hook_ray(origin, point, step):
    o = np.ascontiguousarray(origin, np.float32); q = np.ascontiguousarray(point, np.float32)
    n = C.c_int64(0)
    _lib.lib().sm_debug_mrvm_ray(o.ctypes.data, q.ctypes.data, float(step), None, 0, C.byref(n))
    out = np.zeros((max(n.value, 1), 3), np.int32)
    rc = _lib.lib().sm_debug_mrvm_ray(o.ctypes.data, q.ctypes.data, float(step), out.ctypes.data, n.value, C.byref(n))
    return rc, out[:n.value]


# ---- a restatement of the reference's float / double arithmetic in numpy (cross-check of the tables) ----------
def ref_update(p, hit, hp=0.55, mp=0.48):
    def p2o(x):
        x = np.float32(x)
        return np.float32(np.log(np.float64(x) / (1.0 - np.float64(x))))
    odd = p2o(np.float32(p) / np.float32(256))
    odd = np.float32(odd + (p2o(np.float32(hp)) if hit else p2o(np.float32(mp))))
    prob = np.float32(1.0 - 1.0 / (1.0 + np.float64(np.exp(odd))))
    prob = min(max(prob, np.float32(0.1)), np.float32(0.9))
    return int(np.float32(prob) * np.float32(256))


def test_update_tables_are_the_reference_expressions():
    hit, miss = one_step_tables()
    # p = 0 is never reached (probabilities stay in [25, 230] or 128), and log(0) is where libm and numpy may differ
    for p in range(1, 256):
        assert hit[p] == ref_update(p, True) and miss[p] == ref_update(p, False), p
    assert hit[128] == 140 and miss[128] == 122 and hit[140] == 152   # 0.55, 0.48, then 0.55 again
    assert hit.max() <= 230 and miss.min() >= 25                      # clamp to [0.1, 0.9] * 256


@pytest.mark.parametrize("hp,mp", [(0.55, 0.48), (0.7, 0.4), (0.95, 0.02), (0.501, 0.499)])
def test_binary_lifting_equals_repeated_application(hp, mp):
    hit, miss = one_step_tables(hp, mp)
    rng = np.random.default_rng(5)
    n = 400
    probs = rng.integers(20, 236, n).astype(np.uint8)
    misses = np.concatenate([rng.integers(0, 70, n - 4), [100_000, 2**31 + 7, 2**32 - 1, 0]]).astype(np.int64)
    hits = np.concatenate([rng.integers(0, 70, n - 4), [3, 2**32 - 1, 1, 123_457]]).astype(np.int64)
    got = hook_update(probs, misses, hits, hp, mp)
    for i in range(n):
        p = int(probs[i])
        # a map on 256 values reaches a cycle within 256 steps: iterate the rest modulo the cycle length
        for table, cnt in ((miss, int(misses[i])), (hit, int(hits[i]))):
            seen = {}
            k = 0
            while k < cnt:
                if p in seen:
                    cyc = k - seen[p]
                    k += ((cnt - k) // cyc) * cyc
                    seen = {}
                    if k >= cnt:
                        break
                seen[p] = k
                p = int(table[p])
                k += 1
        assert got[i] == p, i
    # clamped settings give the clamped maps (Initialise, :46-47)
    assert np.array_equal(np.concatenate(one_step_tables(0.95, 0.02)), np.concatenate(one_step_tables(0.9, 0.1)))


# ---- Bresenham: product walk (host hook) == oracle restatement == closed form -----------------------------------
def closed_form_ray(a, b):
    """voxels of the 3-D Bresenham walk in closed form: after t steps an axis with delta d has moved
    max(0, ceil((t d - floor(dm / 2)) / dm)) voxels."""
    a = np.asarray(a, np.int64); b = np.asarray(b, np.int64)
    d = np.abs(b - a); s = np.where(a < b, 1, -1)
    dm = int(d.max())
    if dm == 0:
        return a[None, :].astype(np.int32)
    t = np.arange(dm + 1)[:, None]
    w = np.maximum(0, -((-(t * d[None, :] - (dm >> 1))) // dm))
    return (a[None, :] + s[None, :] * w).astype(np.int32)


def voxel_of(v, step):
    return np.floor(np.asarray(v, np.float32) / np.float32(step)).astype(np.int64)


def test_rays_every_octant_and_long_rays():
    rng = np.random.default_rng(11)
    cases = []
    for sx in (-1, 1):
        for sy in (-1, 1):
            for sz in (-1, 1):
                for _ in range(6):
                    o = rng.uniform(-3, 3, 3)
                    cases.append((o, o + np.array([sx, sy, sz]) * rng.uniform(0, 90, 3)))
    cases += [((0.05, 0.05, 0.05), (0.05, 0.05, 0.05)),                 # point in the origin voxel
              ((0.0, 0.0, 0.0), (80.0, 0.0, 0.0)),                      # axis-aligned, 800 voxels
              ((0.0, 0.0, 0.0), (-55.5, 55.5, -55.5)),                  # diagonal
              ((1.0, 2.0, -3.0), (-1.0e4, 3.7e3, 2.5)),                 # very long (100 000 voxels)
              ((-0.05, -0.15, 0.0), (0.3, -0.3, 0.5))]                  # negative coordinates / borders
    for step in (0.1, 0.5):
        for o, p in cases:
            o = np.float32(o); p = np.float32(p)
            rc, got = hook_ray(o, p, step)
            assert rc == 0
            want = O.voxel_casting_bresenham(o, p, step)
            assert np.array_equal(got, want)
            assert np.array_equal(got, closed_form_ray(voxel_of(o, step), voxel_of(p, step)))
            assert (np.abs(np.diff(got, axis=0)).max(axis=1) == 1).all() if len(got) > 1 else True   # never repeats


def test_ray_hook_refuses_bad_input():
    assert hook_ray((0, 0, 0), (np.nan, 0, 0), 0.1)[0] == -1
    assert hook_ray((0, 0, 0), (2.0e5, 0, 0), 0.1)[0] == -1               # index 2e6 >= 2^20
    assert hook_ray((0, 0, 0), (1.0e5, 0, 0), 0.1)[0] == 0                # index 1e6 < 2^20


# ---- the oracle on hand-computed cases ----------------------------------------------------------------------------
H = {"hit": None, "miss": None}


def tables():
    if H["hit"] is None:
        H["hit"], H["miss"] = one_step_tables()
    return H["hit"], H["miss"]


def state_of(m):
    s = m.State()
    return {int(k): (int(p), int(mi), int(n)) for k, p, mi, n in zip(s["keys"], s["prob"], s["max_intensity"], s["npts"])}


def test_single_ray_and_repeats():
    hit, miss = tables()
    m = O.Mrvm()
    o = (0.05, 0.05, 0.05)
    assert m.InsertPointCloud(pts5([0.55, 0.05, 0.05], 7.9), o) == 0
    assert state_of(m) == {key(5, 0, 0): (hit[128], 7, 1)}
    m.InsertPointCloud(pts5([[0.55, 0.05, 0.05], [0.56, 0.06, 0.01]], [3.0, 12.5]), o)   # two hits, same voxel
    assert state_of(m) == {key(5, 0, 0): (hit[hit[hit[128]]], 12, 3)}
    m.InsertPointCloud(pts5([0.05, 0.05, 0.05], 1.0), o)                 # a point in the origin voxel: only a hit
    assert state_of(m)[key(0, 0, 0)] == (hit[128], 1, 1)
    m.InsertPointCloud(pts5([0.95, 0.05, 0.05]), o)                      # through (0,0,0) and (5,0,0): two misses
    s = state_of(m)
    assert s[key(0, 0, 0)][0] == miss[hit[128]] and s[key(5, 0, 0)][0] == miss[hit[hit[hit[128]]]]


def test_voxel_ended_earlier_and_later_in_the_same_scan():
    hit, miss = tables()
    o = (0.05, 0.05, 0.05)
    A = [0.35, 0.05, 0.05]                                                # voxel (3, 0, 0)
    before = [0.55, 0.05, 0.05]                                           # ray through A, ends at (5, 0, 0)
    after = [0.65, 0.05, 0.05]
    for order, want in (([before, A, after], hit[miss[hit[128]]]),      # miss (need_update), hit, nothing
                        ([A, before, after], hit[hit[128]])):            # hit first: the later rays miss nothing
        m = O.Mrvm()
        m.InsertPointCloud(pts5(A), o)
        m.InsertPointCloud(pts5(order), o)
        assert state_of(m)[key(3, 0, 0)][0] == want
    m = O.Mrvm()                                                          # a voxel born in this scan gets no miss
    m.InsertPointCloud(pts5([A, before]), o)
    assert state_of(m)[key(3, 0, 0)][0] == hit[128]


@pytest.mark.parametrize("max_pts", [1, 10])
def test_stored_points_and_max_intensity(max_pts):
    m = O.Mrvm(max_point_num_in_cell=max_pts)
    xyz = np.array([[0.51 + 0.001 * i, 0.52, 0.53] for i in range(25)], np.float32)
    inten = np.arange(25, dtype=np.float32)[::-1] * 0.5
    m.InsertPointCloud(pts5(xyz[:12], inten[:12]), (0, 0, 0))
    m.InsertPointCloud(pts5(xyz[12:], inten[12:]), (0, 0, 0))
    s = m.State()
    assert s["npts"][0] == max_pts and s["max_intensity"][0] == 12
    assert np.array_equal(s["points"][0, :, :3], xyz[:max_pts])         # the first points by (scan, index)
    avg = O.Mrvm(max_point_num_in_cell=max_pts, output_average=1)
    avg.InsertPointCloud(pts5(xyz, inten), (0, 0, 0))
    out = avg.OutputToPointCloud(0.5)
    acc = np.zeros(3, np.float32)
    for p in xyz[:max_pts]:
        acc = (acc + p).astype(np.float32)
    assert np.array_equal(out[0, :3], acc / np.float32(max_pts)) and out[0, 3] == 12


def test_negative_coordinates_borders_and_z_offset():
    m = O.Mrvm(high_resolution=0.5)
    m.InsertPointCloud(pts5([[-0.1, -0.6, 1.0], [1.0, -1.0, -0.0]]), (0.0, 0.0, 0.0))
    assert sorted(state_of(m)) == sorted([key(-1, -2, 2), key(2, -2, 0)])    # floor, borders belong to the upper voxel
    a, b = O.Mrvm(z_offset=1.0), O.Mrvm()
    b.SetOffsetZ(1.0)
    for mm in (a, b):
        mm.InsertPointCloud(pts5([0.05, 0.05, 0.05]), (0, 0, 0))
        mm.InsertPointCloud(pts5([0.05, 0.05, 2.05]), (0, 0, 0))         # ray from z = 1.0: misses nothing at z = 0
    assert state_of(a) == state_of(b) and state_of(a)[key(0, 0, 0)][0] == tables()[0][128]
    c = O.Mrvm()
    c.InsertPointCloud(pts5([0.05, 0.05, 0.05]), (0, 0, 0))
    c.InsertPointCloud(pts5([0.05, 0.05, 2.05]), (0, 0, 0))             # without the offset the ray starts there
    assert state_of(c)[key(0, 0, 0)][0] == tables()[1][tables()[0][128]]


def test_settings_checks_and_clamps():
    for bad in ({"hit_prob": 0.5}, {"miss_prob": 0.5}, {"max_point_num_in_cell": 0}, {"high_resolution": 0.0}):
        with pytest.raises(ValueError):
            O.Mrvm(**bad)
    rng = np.random.default_rng(2)
    scans = [pts5(rng.uniform(-3, 3, (200, 3))) for _ in range(4)]
    a, b = O.Mrvm(hit_prob=0.97, miss_prob=0.01), O.Mrvm(hit_prob=0.9, miss_prob=0.1)
    for k, s in enumerate(scans):
        a.InsertPointCloud(s, (0.3 * k, 0, 0)); b.InsertPointCloud(s, (0.3 * k, 0, 0))
    assert state_of(a) == state_of(b)


def test_non_finite_dropped_out_of_range_refused_empty_ignored():
    m = O.Mrvm()
    p = pts5([[1, 1, 1], [np.nan, 0, 0], [2, 2, np.inf]])
    assert m.InsertPointCloud(p, (0, 0, 0)) == 2 and m.size() == 1
    before = m.State()
    assert m.InsertPointCloud(pts5([[1, 1, 1], [2.0e5, 0, 0]]), (0, 0, 0)) == -1
    assert m.InsertPointCloud(np.zeros((0, 5), np.float32), (0, 0, 0)) == 0
    after = m.State()
    assert all(np.array_equal(before[k], after[k]) for k in before)


# ---- numpy model of the counting formulation == the serial oracle ----------------------------------------------
class CountingModel:
    """The kernels' formulation: per scan, m(V) = rays j < first_end(V) through V for V born before the scan,
    h(V) = points ending in V; apply m misses, then h hits."""

    def __init__(self, step, max_pts, hit_tab, miss_tab, z_offset=0.0):
        self.step, self.max_pts, self.hit, self.miss, self.z = np.float32(step), max_pts, hit_tab, miss_tab, z_offset
        self.vox = {}      # key tuple -> [prob, max_intensity, points list]

    def insert(self, pts, origin):
        o = np.asarray(origin, np.float32).copy()
        o[2] = np.float32(o[2] + np.float32(self.z))
        ov = voxel_of(o, self.step)
        ok = np.isfinite(pts[:, :3]).all(axis=1)
        idx = np.nonzero(ok)[0]
        ends = voxel_of(pts[idx, :3], self.step)
        first, hits = {}, {}
        for j, e in zip(idx, map(tuple, ends)):
            first.setdefault(e, j)
            hits.setdefault(e, []).append(j)
        old = set(self.vox)
        misses = {}
        for j, e in zip(idx, ends):
            for v in map(tuple, closed_form_ray(ov, e)[:-1]):
                if v in old and j < first.get(v, np.inf):
                    misses[v] = misses.get(v, 0) + 1
        for v in set(misses) | set(hits):
            rec = self.vox.setdefault(v, [128, 0, []])
            for _ in range(misses.get(v, 0)):
                rec[0] = int(self.miss[rec[0]])
            for j in hits.get(v, []):
                rec[0] = int(self.hit[rec[0]])
                rec[1] = max(rec[1], int(pts[j, 3]))
                if len(rec[2]) < self.max_pts:
                    rec[2].append(pts[j, :4].copy())

    def state(self):
        out = {}
        for v, (p, mi, ps) in self.vox.items():
            out[key(*map(int, v))] = (p, mi, len(ps), np.array(ps, np.float32))
        return out


def scene_scans(seed, n_scans, n_pts, extent, step):
    rng = np.random.default_rng(seed)
    scans = []
    for k in range(n_scans):
        xyz = rng.uniform(-extent, extent, (n_pts, 3)).astype(np.float32)
        xyz[: n_pts // 4] = xyz[rng.integers(0, n_pts // 4, n_pts // 4)]           # repeated end voxels
        xyz[n_pts // 4: n_pts // 3] = (np.round(xyz[n_pts // 4: n_pts // 3] / step) * step).astype(np.float32)  # borders
        p = pts5(xyz, rng.uniform(0, 200, n_pts).astype(np.float32))
        p[rng.integers(0, n_pts, 3), rng.integers(0, 3, 3)] = np.nan
        scans.append((p, (0.4 * k - 1.0, 0.1 * k, 0.05)))
    return scans


@pytest.mark.parametrize("seed,max_pts,z", [(0, 10, 0.0), (1, 1, 0.3), (2, 3, -0.2), (3, 10, 0.0)])
def test_counting_model_equals_serial_oracle(seed, max_pts, z):
    step = 0.25
    hit, miss = tables()
    model = CountingModel(step, max_pts, hit, miss, z)
    orc = O.Mrvm(high_resolution=step, max_point_num_in_cell=max_pts, z_offset=z)
    for pts, origin in scene_scans(seed, 6, 300, 2.0, step):
        model.insert(pts, origin)
        assert orc.InsertPointCloud(pts, origin) == 3
    want = orc.State()
    got = model.state()
    assert sorted(got) == [int(k) for k in want["keys"]]
    for i, k in enumerate(want["keys"]):
        p, mi, n, ps = got[int(k)]
        assert (p, mi, n) == (int(want["prob"][i]), int(want["max_intensity"][i]), int(want["npts"][i]))
        assert np.array_equal(ps.view(np.uint32), want["points"][i, :n].view(np.uint32))
    assert len(set(int(x) for x in want["prob"])) > 5          # the scenes exercise many probability levels
