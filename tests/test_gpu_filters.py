"""The filter chain (pre_processers::filter::Factory and its nine filters) on the GPU against the serial oracle: every
filter alone and the shipped chains on full-size synthetic scans, bit for bit; RandomSampler determinism; the edge
cases of a call; the device path; and filter -> motion compensation -> MultiResolutionVoxelMap without a host round
trip."""
import ctypes as C

import numpy as np
import pytest

import filters_oracle as O
import staticmapping_b200 as smb
from staticmapping_b200 import _lib, synth

pytestmark = pytest.mark.gpu

F, I = 1, 0
CHAINS = {
    "Range": [("Range", {"min_range": (F, "4.5"), "max_range": (F, "75")})],
    "AxisRange": [("AxisRange", {"min": (F, "-1.2"), "max": (F, "2."), "axis_index": (I, "2")})],
    "BoundingBoxRemoval": [("BoundingBoxRemoval", {"min_x": (F, "-3"), "max_x": (F, "3"), "min_y": (F, "-2"),
                                                   "max_y": (F, "2"), "min_z": (F, "-5"), "max_z": (F, "5")})],
    "RandomSampler": [("RandomSampler", {"sampling_rate": (F, "0.35")})],
    "StatisticRemoval": [("StatisticRemoval", {})],
    "RangeImage": [("RangeImage", {"top_angle": (F, "3"), "btm_angle": (F, "-25"), "vertical_line_num": (I, "64"),
                                   "horizontal_line_num": (I, "900")})],
    "GroundRemoval": [("GroundRemoval", {"leaf_size": (F, "0.8"), "height_threshold": (F, "0.15")})],
    "GroundRemoval2": [("GroundRemoval2", {"r_min": (F, "0.1"), "start_ground_height": (F, "-1.5"),
                                           "long_line_threshold": (F, "10"), "max_slope": (F, "0.12"),
                                           "max_error": (F, "0.1"), "max_dist_to_line": (F, "0.10"),
                                           "max_start_height": (F, "0.6"), "thread_num": (I, "4")})],
    "VoxelGrid": [("VoxelGrid", {"voxel_size": (F, "0.2")})],
}
CHAINS["default_xml"] = [CHAINS["Range"][0], CHAINS["RandomSampler"][0]]
CHAINS["kitti_xml"] = [("Range", {"min_range": (F, "5.")}), ("AxisRange", {"min": (F, "-2.")}),
                       ("RandomSampler", {"sampling_rate": (F, "0.5")})]
CHAINS["ground2_rangeimage_voxel"] = [CHAINS["Range"][0], CHAINS["RangeImage"][0], CHAINS["GroundRemoval2"][0],
                                      CHAINS["RandomSampler"][0], CHAINS["VoxelGrid"][0]]


def scans(n=10):
    scene = synth.make_scene(seed=5)
    out = []
    for k in range(n):
        p = synth.lidar_scan(scene, (0.5 * k, 0.0, 0.0), seed=100 + k)
        r = np.zeros((p.shape[0], 5), np.float32)
        r[:, :3] = p
        r[:, 3] = np.random.default_rng(k).uniform(0, 100, p.shape[0])
        r[:, 4] = np.linspace(0, 1, p.shape[0], dtype=np.float32)
        out.append(r)
    return out


_SCANS = scans()


def gpu_chain(stages, seed=0):
    c = smb.FilterChain(0)
    c.set_seed(seed)
    for name, params in stages:
        k = c.add(name)
        assert k >= 0
        for pname, (t, text) in params.items():
            assert c.set_param(k, pname, t, text) == 0
    return c


@pytest.mark.parametrize("chain", list(CHAINS))
def test_chain_bit_identical_to_oracle(chain):
    g = gpu_chain(CHAINS[chain], seed=7)
    o = O.Chain(O.ANGLE_PRODUCT)
    o.set_seed(7)
    for name, params in CHAINS[chain]:
        k = o.add(name)
        for pname, (t, text) in params.items():
            o.set_param(k, pname, t, text)
    for pts in _SCANS:
        rc, out, kept = g.filter(pts)
        orc, oout, okept = o.filter(pts)
        assert rc == 0 and orc == 0
        assert out.shape == oout.shape, (chain, out.shape, oout.shape)
        np.testing.assert_array_equal(kept, okept)
        assert out.tobytes() == oout.tobytes()
        np.testing.assert_array_equal(g.stage_counts(), o.stage_counts())
    print(f"{chain}: {pts.shape[0]} -> {out.shape[0]} points, stage counts {list(g.stage_counts())}")


@pytest.mark.parametrize("chain", ["RangeImage", "GroundRemoval2"])
def test_host_atan2f_differences_are_reported(chain):
    """against the literal reference (host atan2f) only points on a pixel / cell border may differ"""
    g = gpu_chain(CHAINS[chain])
    differ = 0
    for pts in _SCANS[:3]:
        _, _, kept = g.filter(pts)
        _, _, okept = O.run_chain(CHAINS[chain], pts, angle_mode=O.ANGLE_HOST)
        differ += len(np.setxor1d(kept, okept))
    print(f"{chain}: {differ} of {3 * _SCANS[0].shape[0]} points differ from a host-atan2f run")
    assert differ < 0.01 * 3 * _SCANS[0].shape[0]


def test_random_sampler_determinism():
    st = CHAINS["RandomSampler"]
    pts = _SCANS[0]
    a = gpu_chain(st, seed=11); b = gpu_chain(st, seed=11); c = gpu_chain(st, seed=12)
    ra, rb, rc = a.filter(pts), b.filter(pts), c.filter(pts)
    assert ra[1].tobytes() == rb[1].tobytes() and np.array_equal(ra[2], rb[2])
    assert not np.array_equal(ra[2][:1000], rc[2][:1000])
    nxt = a.filter(pts)
    assert not np.array_equal(nxt[2][:1000], ra[2][:1000])
    n = pts.shape[0]
    for r in (ra, rc, nxt):                       # binomial: 6 sigma
        assert abs(r[1].shape[0] - 0.35 * n) < 6 * np.sqrt(n * 0.35 * 0.65)


def test_edge_cases():
    c = gpu_chain(CHAINS["default_xml"])
    rc, out, kept = c.filter(np.zeros((0, 5), np.float32))
    assert rc == 0 and out.shape == (0, 5)
    # a chain that removes every point, then more stages
    e = gpu_chain([("BoundingBoxRemoval", {}), ("RangeImage", {}), ("GroundRemoval", {}), ("VoxelGrid", {})])
    rc, out, kept = e.filter(_SCANS[0])
    assert rc == 0 and out.shape == (0, 5) and list(e.stage_counts()) == [0, 0, 0, 0]
    # non-finite points
    p = _SCANS[1][:5000].copy()
    p[::7, 0] = np.nan
    p[::11, 2] = np.inf
    for chain in ("Range", "AxisRange", "RangeImage", "GroundRemoval", "GroundRemoval2", "VoxelGrid"):
        g = gpu_chain(CHAINS[chain])
        r = g.filter(p)
        o = O.run_chain(CHAINS[chain], p)
        assert r[0] == 0 and r[1].tobytes() == o[1].tobytes() and np.array_equal(r[2], o[2]), chain
    # an invalid stage: SM_ERR_BAD_ARGUMENT and nothing written
    bad = gpu_chain([("AxisRange", {"min": (F, "3"), "max": (F, "1")})])
    out = np.full((10, 5), 7.0, np.float32)
    m = C.c_int64(0)
    pts = np.ascontiguousarray(_SCANS[0][:10])
    rc = _lib.lib().sm_filter_chain_filter(bad._h, pts.ctypes.data, 10, 20, out.ctypes.data, 10, C.byref(m), None)
    assert rc == -1 and (out == 7.0).all()
    # too small a capacity: the count is reported, the output untouched
    ok = gpu_chain(CHAINS["Range"])
    rc = _lib.lib().sm_filter_chain_filter(ok._h, pts.ctypes.data, 10, 20, out.ctypes.data, 1, C.byref(m), None)
    assert rc == -1 and m.value > 1 and (out == 7.0).all()


def test_device_path_equals_host_path_and_feeds_the_map():
    import torch
    st = CHAINS["default_xml"]
    host = gpu_chain(st, seed=3)
    dev = gpu_chain(st, seed=3)
    delta = np.eye(4)
    delta[:3, 3] = [0.3, -0.1, 0.02]
    a = np.deg2rad(2.0)
    delta[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
    m_host = smb.MultiResolutionVoxelMap(0)
    m_dev = smb.MultiResolutionVoxelMap(0)
    m_host.Initialise(smb.MrvmSettings())
    m_dev.Initialise(smb.MrvmSettings())
    lib = _lib.lib()
    d = np.asfortranarray(delta)
    f = smb.FilterFactory(0, seed=3, chain=dev)
    for k, pts in enumerate(_SCANS[:4]):
        origin = np.array([0.5 * k, 0.0, 0.0], np.float32)
        rc, out, kept = host.filter(pts)
        assert rc == 0
        comp = smb.MotionCompensation(out, delta)
        m_host.InsertPointCloud(comp, origin)
        # device: one upload, then everything stays on the GPU
        t = torch.from_numpy(pts).cuda()
        torch.cuda.synchronize()
        out_d, kept_d = f.FilterDevice(t)
        assert out_d.cpu().numpy().tobytes() == out.tobytes() and np.array_equal(kept_d.cpu().numpy(), kept)
        comp_d = torch.empty_like(out_d)
        stream = torch.cuda.current_stream().cuda_stream
        assert lib.sm_motion_compensation_device(0, out_d.data_ptr(), out_d.shape[0], 20, d.ctypes.data_as(_lib._DP),
                                                 comp_d.data_ptr(), stream) == 0
        m_dev.InsertPointCloud(comp_d, origin)
    a, b = m_host.State(), m_dev.State()
    for key in a:
        assert a[key].tobytes() == b[key].tobytes(), key


def test_python_classes_on_the_gpu():
    pts = _SCANS[2]
    r = smb.Range(0)
    assert r.InitFromXmlText('<filter name="Range"><param type="1" name="min_range">4.5</param></filter>')
    r.SetInputCloud(pts)
    out = r.Filter()
    o = smb.Range(chain=O.Chain())
    o.InitFromXmlText('<filter name="Range"><param type="1" name="min_range">4.5</param></filter>')
    o.SetInputCloud(pts)
    assert out.tobytes() == o.Filter().tobytes()
    assert np.array_equal(r.Inliers(), o.Inliers()) and np.array_equal(r.Outliers(), o.Outliers())
    g = smb.GroundRemoval(0)
    g.SetInputCloud(pts)
    out = g.Filter()
    assert len(g.Inliers()) == out.shape[0] and len(g.Outliers()) > 0
    assert len(g.Inliers()) + len(g.Outliers()) <= pts.shape[0]


def test_cpp_adapter_end_to_end(tmp_path):
    import os
    import shutil
    import struct
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if cxx is None:
        pytest.skip("no g++")
    libdir = os.path.join(root, "staticmapping_b200")
    exe = str(tmp_path / "filters_run")
    r = subprocess.run([cxx, "-std=c++14", "-O1", "-Wall", "-I", os.path.join(root, "tests", "stubs"), "-I",
                        os.path.join(root, "include"), "-I", os.path.join(root, "adapter"),
                        os.path.join(root, "tests", "cpp", "filters_run.cc"), "-o", exe, "-L", libdir,
                        "-l:libsm_b200.so", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    with open(tmp_path / "in.bin", "wb") as f:
        f.write(struct.pack("<q", 3))
        for pts in _SCANS[:3]:
            f.write(struct.pack("<q", pts.shape[0]))
            f.write(pts.tobytes())
    r = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    raw = open(tmp_path / "out.bin", "rb").read()
    o = O.Chain()
    o.set_seed(7)
    for name, params in CHAINS["default_xml"]:
        k = o.add(name)
        for pname, (t, text) in params.items():
            o.set_param(k, pname, t, text)
    pos = 0
    for pts in _SCANS[:3]:
        m = struct.unpack_from("<q", raw, pos)[0]
        pos += 8
        got = raw[pos:pos + 20 * m]
        pos += 20 * m
        assert got == o.filter(pts)[1].tobytes()
