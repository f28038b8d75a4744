"""CPU checks of the filter chain (pre_processers::filter::Factory and its nine filters): the serial oracle on
hand-computed cases, the reference's own unit tests (pre_processors/test/test_filter_*.cc) replayed through the Python
classes on the oracle, numpy models of the GPU formulations against the oracle, and the product's host-compiled
per-point functions and FitLines (include/sm_b200_debug.h) against the oracle."""
import ctypes as C

import numpy as np
import pytest

import filters_oracle as O
import staticmapping_b200 as smb
from staticmapping_b200 import _lib, synth

F, I = 1, 0


def rec(xyz):
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    r = np.zeros((xyz.shape[0], 5), np.float32)
    r[:, :3] = xyz
    return r


def run(stages, pts, **kw):
    rc, out, kept = O.run_chain(stages, rec(pts) if np.asarray(pts).shape[-1] == 3 else pts, **kw)
    assert rc == 0
    return out, kept


def scan(seed=0):
    scene = synth.make_scene(seed=5)
    p = synth.lidar_scan(scene, (0.0, 0.0, 0.0), seed=100 + seed)
    r = rec(p)
    r[:, 4] = np.linspace(0, 1, p.shape[0], dtype=np.float32)
    return r


# ---- 1. the oracle on hand-computed cases ----------------------------------------------------------------------
def test_nan_kept_by_axis_range_removed_by_range():
    pts = [[np.nan, 0, 0], [0, 0, 10], [0, 0, 1]]
    _, kept = run([("AxisRange", {"min": (F, "-5"), "max": (F, "5"), "axis_index": (I, "0")})], pts)
    assert list(kept) == [0, 1, 2]
    _, kept = run([("Range", {"min_range": (F, "0.5"), "max_range": (F, "5")})], pts)
    assert list(kept) == [2]
    # AxisRange at its defaults is the identity (inf kept); an explicit FLT_MAX bound drops +inf
    _, kept = run([("AxisRange", {})], [[0, 0, np.inf]])
    assert list(kept) == [0]
    _, kept = run([("AxisRange", {"min": (F, "-1e30")})], [[0, 0, np.inf], [0, 0, 1]])
    assert list(kept) == [1]


def test_range_image_row_zero_below_btm_and_first_point_wins():
    # V = 10 rows over [-10, 10] degrees: 2 degrees a row; a point 0.3 rows (0.6 deg) below btm lands in row 0
    st = [("RangeImage", {"top_angle": (F, "10"), "btm_angle": (F, "-10"), "vertical_line_num": (I, "10"),
                          "horizontal_line_num": (I, "360")})]
    d = 10.0
    below = [d, 0, d * np.tan(np.deg2rad(-10.6))]
    far_below = [d, 0, d * np.tan(np.deg2rad(-12.5))]
    _, kept = run(st, [below, far_below])
    assert list(kept) == [0]
    # the same pixel twice: the first in input order is the inlier; xy < 0.01 is an outlier
    _, kept = run(st, [[0.005, 0, 0], [d, 0.001, 0], [d, 0, 0.0001], [d, 5, 0]])
    assert list(kept) == [1, 3]


def test_ground_removal_small_voxel_vanishes_and_ground_is_removed():
    st = [("GroundRemoval", {"leaf_size": (F, "1"), "min_point_num_in_voxel": (I, "3")})]
    flat = [[0.5, 0.5, -0.5 + 0.01 * k] for k in range(4)]            # voxel (0,0,0): delta 0.03 -> ground
    tall = [[2.5, 0.5, -0.9], [2.5, 0.5, -0.1], [2.5, 0.6, -0.5]]     # voxel (2,0,0): delta 0.8 -> kept
    lone = [[5.5, 0.5, -0.5], [5.5, 0.5, -0.4]]                        # 2 < 3 points: vanishes
    high = [[-1.5, 0.5, 1.5]] * 3                                      # voxel (-1,0,1): iz > 0 -> kept
    out, kept = run(st, flat + tall + lone + high)
    # std::map order: (-1,0,1) before (2,0,0)
    assert list(kept) == [9, 10, 11, 4, 5, 6]
    g = smb.GroundRemoval(chain=O.Chain())
    assert g.InitFromXmlText('<filter name="GroundRemoval"><param type="1" name="leaf_size">1</param>'
                             '<param type="0" name="min_point_num_in_voxel">3</param></filter>')
    g.SetInputCloud(rec(flat + tall + lone + high))
    g.Filter()
    assert list(g.Inliers()) == [4, 5, 6, 9, 10, 11] and list(g.Outliers()) == [0, 1, 2, 3]


def test_statistic_removal_is_the_identity_even_first():
    pts = rec(np.random.default_rng(0).normal(size=(50, 3)))
    out, kept = run([("StatisticRemoval", {}), ("Range", {"max_range": (F, "1.5")})], pts)
    out2, kept2 = run([("Range", {"max_range": (F, "1.5")})], pts)
    assert np.array_equal(kept, kept2) and out.tobytes() == out2.tobytes()


def test_ground_removal2_farthest_candidate_segment_first():
    """a point whose own segment has no line takes the first positive distance of +step, -step, ... +1, -1"""
    B, S = 20, 36                                                    # 10-degree segments, 5 m bins over 0-100 m
    kw = dict(r_min=0.0, r_max=100.0, bin_num=B, segment_num=S, search_angle=20.0, max_start_height=10.0,
              start_ground_height=0.0, max_error=1.0, max_slope=1.0, long_line_threshold=100.0)
    def ray(deg, z0, slope):
        a = np.deg2rad(deg)
        d = 2.5 + 5.0 * np.arange(6)
        return np.stack([d * np.cos(a), d * np.sin(a), z0 + slope * d], 1)
    pts = np.concatenate([ray(25, 0.0, 0.0), ray(-15, 0.3, 0.0), ray(5, 0.0, 0.0)[:1]])
    # segment 2 (20-30 deg): line z = 0; segment 34 (-20..-10 deg): line z = 0.3; segment 0 has one point: no line
    st = O.gr2_state(rec(pts), **kw)
    assert st["nlines"][2] == 1 and st["nlines"][34] == 1 and st["nlines"][0] == 0
    # the query point in segment 0 at z = 0.04: step 2 first -> segment 2 (distance 0.04 <= 0.05) -> ground
    stages = [("GroundRemoval2", {k: (F if isinstance(v, float) else I, str(v)) for k, v in kw.items()})]
    stages[0][1]["max_dist_to_line"] = (F, "0.05")
    q = rec(np.concatenate([pts, [[7.5 * np.cos(np.deg2rad(5)), 7.5 * np.sin(np.deg2rad(5)), 0.04]]]))
    _, kept = run(stages, q)
    assert q.shape[0] - 1 not in kept
    # the same point at z = 0.26: segment 2 gives 0.26 > 0.05 (first positive distance wins) -> not ground,
    # although segment 34 (step -2, tried after +2) would have matched
    q[-1, 2] = 0.26
    _, kept = run(stages, q)
    assert q.shape[0] - 1 in kept


# ---- 2. the reference's unit tests, through the Python classes on the oracle -------------------------------------
def test_filter_config_cases():
    ax = smb.AxisRange(chain=O.Chain())
    assert not ax.InitFromXmlText('<filter name="AxisRange"><param type="1" name="min">1</param>'
                                  '<param type="1" name="max">-1</param></filter>')
    assert not ax.InitFromXmlText('<filter name="AxisRange"><param type="1" name="min">-1</param>'
                                  '<param type="1" name="max">1</param><param type="0" name="axis_index">3</param>'
                                  '</filter>')
    assert not ax.InitFromXmlText('<filter name="AxisRange"><param type="0" name="axis_index">-1</param></filter>')
    bb = smb.BoundingBoxRemoval(chain=O.Chain())
    assert not bb.InitFromXmlText('<filter name="BoundingBoxRemoval"><param type="1" name="min_x">1</param>'
                                  '<param type="1" name="max_x">-1</param></filter>')
    rs = smb.RandomSampler(chain=O.Chain())
    assert rs.InitFromXmlText('<filter name="RandomSampler"><param type="1" name="sampling_rate">0.5</param></filter>')
    assert not rs.InitFromXmlText('<filter name="RandomSampler"><param type="1" name="sampling_rate">1.5</param>'
                                  '</filter>')
    assert rs.InitFromXmlText('<filter name="RandomSampler"><param type="1" name="sampling_rate">0.</param></filter>')
    assert not rs.InitFromXmlText('<filter name="RandomSampler"><param type="1" name="sampling_rate">-0.1</param>'
                                  '</filter>')
    vg = smb.VoxelGrid(chain=O.Chain())
    assert not vg.InitFromXmlText('<filter name="VoxelGrid"><param type="1" name="voxel_size">0.</param></filter>')
    assert vg.InitFromXmlText('<filter name="VoxelGrid"><param type="1" name="voxel_size">0.1</param></filter>')
    # another filter's node: false; an unknown parameter or type: the reference's CHECK failure
    assert not vg.InitFromXmlText('<filter name="Range"><param type="1" name="min_range">1</param></filter>')
    with pytest.raises(smb.CheckFailure):
        vg.InitFromXmlText('<filter name="VoxelGrid"><param type="1" name="leaf">0.1</param></filter>')
    with pytest.raises(smb.CheckFailure):
        vg.InitFromXmlText('<filter name="VoxelGrid"><param name="voxel_size">0.1</param></filter>')
    f = smb.FilterFactory(chain=O.Chain())
    with pytest.raises(smb.CheckFailure):
        f.InitFromXmlText('<filters><filter name="NoSuchFilter"/></filters>')


def test_range_axis_range_bounding_box_assertions():
    rng = np.random.default_rng(1)
    cloud = rec(rng.uniform(0, 100, (10000, 3)))
    r = smb.Range(chain=O.Chain())
    r.SetInputCloud(cloud)
    assert r.Filter().shape[0] == cloud.shape[0]                     # identity at defaults
    assert r.InitFromXmlText('<filter name="Range"><param type="1" name="min_range">20</param>'
                             '<param type="1" name="max_range">80</param></filter>')
    out = r.Filter()
    d = np.sqrt((out[:, :3].astype(np.float32) ** 2).sum(1))
    assert (d >= 20).all() and (d <= 80).all() and len(r.Inliers()) + len(r.Outliers()) == cloud.shape[0]
    ax = smb.AxisRange(chain=O.Chain())
    ax.SetInputCloud(cloud)
    assert ax.Filter().shape[0] == cloud.shape[0]
    assert ax.InitFromXmlText('<filter name="AxisRange"><param type="1" name="min">10</param></filter>')
    assert ax.InitFromXmlText('<filter name="AxisRange"><param type="1" name="max">60</param></filter>')
    out = ax.Filter()                                                # min = 10 persists from the first call
    assert out.shape[0] > 0 and (out[:, 2] >= 10).all() and (out[:, 2] <= 60).all()
    assert ax.InitFromXmlText('<filter name="AxisRange"><param type="0" name="axis_index">0</param></filter>')
    out = ax.Filter()
    assert (out[:, 0] >= 10).all() and (out[:, 0] <= 60).all()
    bb = smb.BoundingBoxRemoval(chain=O.Chain())
    bb.SetInputCloud(cloud)
    assert bb.Filter().shape[0] == 0                                 # the default box removes everything finite
    assert bb.InitFromXmlText('<filter name="BoundingBoxRemoval">' + "".join(
        f'<param type="1" name="{k}">{v}</param>' for k, v in
        [("min_x", 0), ("min_y", 0), ("min_z", 0), ("max_x", 100), ("max_y", 100), ("max_z", 100)]) + '</filter>')
    assert bb.Filter().shape[0] == 0
    assert bb.InitFromXmlText('<filter name="BoundingBoxRemoval"><param type="1" name="max_x">50</param></filter>')
    out = bb.Filter()
    assert out.shape[0] > 0 and (out[:, 0] > 50).all()


def test_random_sampler_fraction_and_identity():
    cloud = rec(np.random.default_rng(2).uniform(-1, 1, (100000, 3)))
    rs = smb.RandomSampler(chain=O.Chain(), seed=5)
    assert rs.InitFromXmlText('<filter name="RandomSampler"><param type="1" name="sampling_rate">0.5</param>'
                              '</filter>')
    rs.SetInputCloud(cloud)
    sizes = [rs.Filter().shape[0] / cloud.shape[0] for _ in range(100)]
    assert all(0.48 < s < 0.52 for s in sizes) and len(set(sizes)) > 50
    assert rs.InitFromXmlText('<filter name="RandomSampler"><param type="1" name="sampling_rate">0.9995</param>'
                              '</filter>')
    assert rs.Filter().shape[0] == cloud.shape[0]


# ---- 3. numpy models of the GPU formulations -------------------------------------------------------------------
def debug_points(op, pts, params, width=1):
    p = np.ascontiguousarray(pts, np.float32)
    out = np.zeros(p.shape[0] * width, np.int64)
    prm = np.ascontiguousarray(params, np.float32)
    assert _lib.lib().sm_debug_filter_points(op, p.ctypes.data, p.shape[0], 4 * p.shape[1], prm.ctypes.data,
                                             out.ctypes.data) == 0
    return out.reshape(-1, width) if width > 1 else out


RI = ("RangeImage", {"top_angle": (F, "3"), "btm_angle": (F, "-25"), "vertical_line_num": (I, "64"),
                     "horizontal_line_num": (I, "900")})


def test_range_image_min_index_per_pixel_equals_oracle():
    pts = scan(1)
    pix = debug_points(1, pts, [3, -25, 0, 0, 0, 64, 900])           # the product's pixel function
    valid = pix >= 0
    first = {}
    for i in np.flatnonzero(valid):                                  # atomicMin of the index per pixel
        first.setdefault(pix[i], i)
    model = np.sort(np.array(list(first.values())))
    _, kept = run([RI], pts)
    assert np.array_equal(model, kept)


def test_ground_removal_sorted_keys_equal_map_order():
    pts = scan(2)
    st = [("GroundRemoval", {"leaf_size": (F, "0.8")})]
    _, kept = run(st, pts)
    v = debug_points(3, pts, [0.8], width=4)
    assert (v[:, 0] == 0).all()
    order = np.lexsort((np.arange(pts.shape[0]), v[:, 3], v[:, 2], v[:, 1]))   # stable sort by (ix, iy, iz)
    keys = v[order, 1:]
    head = np.r_[True, (keys[1:] != keys[:-1]).any(1)]
    seg = np.cumsum(head) - 1
    cnt = np.bincount(seg)
    z = pts[order, 2]
    zmax = np.full(cnt.size, -1e9, np.float32); np.maximum.at(zmax, seg, z)
    zmin = np.full(cnt.size, 1e9, np.float32); np.minimum.at(zmin, seg, z)
    iz = keys[head][:, 2]
    ground = (iz <= 0) & ((zmax - zmin) >= 0) & ((zmax - zmin) <= np.float32(0.15))
    keep = (cnt >= 10) & ~ground
    assert np.array_equal(order[keep[seg]], kept)


def test_ground_removal2_segmented_running_min_membership():
    pts = scan(3)
    st = O.gr2_state(pts)
    cell = debug_points(2, pts, [100, 1, 200, 180])
    assert np.array_equal(cell, st["cell"])                          # product host build == oracle, bit for bit
    order = np.argsort(cell, kind="stable")
    c = cell[order]
    z = pts[order, 2]
    member = np.zeros(pts.shape[0], np.uint8)
    start = np.r_[0, np.flatnonzero(c[1:] != c[:-1]) + 1, c.size]
    for a, b in zip(start[:-1], start[1:]):                          # running minimum inside each cell
        run_min = np.minimum.accumulate(z[a:b])
        member[order[a:b]] = (z[a:b].astype(np.float64) <= run_min.astype(np.float64) + 0.5)
    assert np.array_equal(member, st["member"])


# ---- 4. the product's host build against the oracle ------------------------------------------------------------
def test_angle_and_pixel_functions_bit_identical_in_product_mode():
    pts = scan(4)
    a = debug_points(0, pts, [0]).astype(np.uint32).view(np.float32)
    ref = np.arctan2(pts[:, 1].astype(np.float64), pts[:, 0].astype(np.float64))
    assert np.abs(a.astype(np.float64) - ref).max() < 4e-7           # a float-accurate atan2
    edge = rec([[0, 0, 0], [1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [-1, -1e-30, 0], [np.inf, 1, 0]])
    e = debug_points(0, edge, [0]).astype(np.uint32).view(np.float32)
    assert np.array_equal(e, np.float32([0, 0, np.pi, np.pi / 2, -np.pi / 2, -np.pi, 0]))


def test_host_atan2f_differences_lie_on_cell_borders():
    """the literal reference (host atan2f) bins a point elsewhere only when its angle quotient is within 4 float ulps
    of a segment border"""
    pts = scan(5)
    a = O.gr2_state(pts, angle_mode=O.ANGLE_PRODUCT)["cell"]
    b = O.gr2_state(pts, angle_mode=O.ANGLE_HOST)["cell"]
    diff = np.flatnonzero(a != b)
    print(f"{diff.size} of {pts.shape[0]} points in another cell with the host atan2f")
    rad = debug_points(0, pts[diff], [0]).astype(np.uint32).view(np.float32)
    rad = np.where(rad < 0, rad + np.float32(2 * np.pi), rad).astype(np.float32)
    q = rad / np.float32(2 * np.pi / 180)
    assert (np.abs(q - np.round(q)) <= 4 * np.spacing(np.abs(q).astype(np.float32))).all()
    assert ((a[diff] // 200) != (b[diff] // 200)).all()              # only the segment moves, never the bin


def test_fit_lines_equal_oracle():
    kw = dict(r_min=0.1, start_ground_height=-1.5, long_line_threshold=10.0, max_slope=0.12, max_error=0.1,
              max_dist_to_line=0.1, max_start_height=0.6)                # lidar_only_kitti.xml's GroundRemoval2
    P = dict(O.GR2_DEFAULTS, **kw)
    params = np.array([P[k] for k in O.GR2_ORDER[:-1]], np.float32)
    for seed in range(3):
        pts = scan(6 + seed)
        st = O.gr2_state(pts, **kw)
        checked = 0
        for s in range(180):
            dz = np.ascontiguousarray(st["cell_dz"][s * 200:(s + 1) * 200])
            used = np.ascontiguousarray(st["cell_used"][s * 200:(s + 1) * 200])
            lines = np.zeros((102, 4), np.float32)
            n = C.c_int64(0)
            assert _lib.lib().sm_debug_filter_fit_lines(dz.ctypes.data, used.ctypes.data, params.ctypes.data,
                                                        lines.ctypes.data, 102, C.byref(n)) == 0
            assert n.value == st["nlines"][s]
            ol = st["lines"][s, :n.value]
            np.testing.assert_array_max_ulp(lines[:n.value], ol, maxulp=1)
            checked += n.value
        assert checked > 50


def test_line_fit_matches_least_squares():
    rng = np.random.default_rng(9)
    for k in (2, 3, 7, 40):
        d = np.sort(rng.uniform(1, 80, k)).astype(np.float32)
        z = (0.02 * d - 1.7 + rng.normal(0, 0.01, k)).astype(np.float32)
        dz = np.ascontiguousarray(np.stack([d, z], 1))
        mb = np.zeros(3, np.float32)
        assert _lib.lib().sm_debug_filter_line_fit(dz.ctypes.data, k, mb.ctypes.data) == 0
        m, b = np.linalg.lstsq(np.stack([d.astype(np.float64), np.ones(k)], 1), z.astype(np.float64), rcond=None)[0]
        assert abs(mb[0] - m) <= 2e-6 * max(1, abs(m)) + 1e-7 and abs(mb[1] - b) <= 2e-6 * max(1, abs(b))
        err = np.abs(np.float32(mb[0]) * d + np.float32(mb[1]) - z).max()
        assert mb[2] == err


def test_factory_runs_the_shipped_chains_on_the_oracle():
    pts = scan(10)
    f = smb.FilterFactory(chain=O.Chain(), seed=1)
    f.InitFromXmlText('<filters><filter name="Range"><param type="1" name="min_range">4.5</param>'
                      '<param type="1" name="max_range">75</param></filter>'
                      '<filter name="RandomSampler"><param type="1" name="sampling_rate">0.35</param></filter>'
                      '</filters>')
    f.SetInputCloud(pts)
    out = f.Filter()
    c = f.StageCounts()
    assert c[1] == out.shape[0] and 0.3 * c[0] < c[1] < 0.4 * c[0]
    e = smb.FilterFactory(chain=O.Chain())
    e.InitFromXmlText("<filters/>")
    e.SetInputCloud(pts)
    assert e.Filter().tobytes() == pts.tobytes()                     # an empty chain copies its input
