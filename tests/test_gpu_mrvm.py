"""MultiResolutionVoxelMap on the GPU against the serial oracle: full-size lidar sequences bit for bit (state and every
output form), determinism, table growth, the edge cases of an insert, device inserts, a moving object removed from
the static map, and the C++ adapter end to end."""
import os
import shutil
import struct
import subprocess

import numpy as np
import pytest

import mrvm_oracle as O
import staticmapping_b200 as smb
from staticmapping_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOX_LO, BOX_HI = np.array([4.0, 1.0, -1.73]), np.array([5.0, 1.8, -0.73])   # beside the sensor track, 1 m tall


def scan(k, scene, seed_base=0):
    """full-size scan (120 000 points) from (k, 0, 0) in the world frame, InnerPointType rows"""
    pos = np.array([float(k), 0.0, 0.0])
    p = synth.lidar_scan(scene, pos, seed=seed_base + k)
    pts = np.zeros((p.shape[0], 5), np.float32)
    pts[:, :3] = p + pos.astype(np.float32)
    pts[:, 3] = np.random.default_rng(k).uniform(0, 180, p.shape[0]).astype(np.float32)
    pts[:, 4] = np.linspace(0, 1, p.shape[0], dtype=np.float32)
    return pts, pos


_SCANS = {}


def sequence(n=10):
    if n not in _SCANS:
        scene = synth.make_scene(seed=3)
        _SCANS[n] = [scan(k, scene) for k in range(n)]
    return _SCANS[n]


def gpu_map(expected_voxels=1 << 20, **kw):
    m = smb.MultiResolutionVoxelMap(expected_voxels=expected_voxels)
    m.Initialise(smb.MrvmSettings(**kw))
    return m


def same_state(a, b):
    return all(np.array_equal(a[k], b[k]) for k in ("keys", "prob", "max_intensity", "npts")) and \
        np.array_equal(a["points"].view(np.uint32), b["points"].view(np.uint32))


@pytest.mark.parametrize("average,use_max", [(0, 1), (1, 1), (0, 0), (1, 0)])
def test_full_size_sequence_bit_identical(average, use_max):
    g = gpu_map(expected_voxels=1000, output_average=average, use_max_intensity=use_max)   # grows far past 1000
    o = O.Mrvm(output_average=average, use_max_intensity=use_max)
    for pts, pos in sequence():
        assert g.InsertPointCloud(pts, pos) == 0 and o.InsertPointCloud(pts, pos) == 0
    assert g.size() == o.size() > 100 * 1000
    assert same_state(g.State(), o.State())
    for thr in (0.5, 0.6, 0.57):
        for rgb in (0, 1):
            want = o.OutputToPointCloud(thr, rgb)
            got = g.OutputToPointCloud(thr, rgb)
            assert got.shape == want.shape and np.array_equal(got.view(np.uint32), want.view(np.uint32)), (thr, rgb)


def test_two_runs_identical_bytes():
    outs = []
    for _ in range(2):
        g = gpu_map()
        for pts, pos in sequence()[:5]:
            g.InsertPointCloud(pts, pos)
        outs.append((g.OutputToPointCloud(0.5).tobytes(), g.State()))
    assert outs[0][0] == outs[1][0] and same_state(outs[0][1], outs[1][1])


def test_empty_cloud_non_finite_and_out_of_range():
    pts, pos = sequence()[0]
    g = gpu_map(hit_prob=0.7, miss_prob=0.4, max_point_num_in_cell=1, z_offset=0.35)
    o = O.Mrvm(hit_prob=0.7, miss_prob=0.4, max_point_num_in_cell=1, z_offset=0.35)
    assert g.InsertPointCloud(pts, pos) == 0 and o.InsertPointCloud(pts, pos) == 0
    before = g.State()
    assert g.InsertPointCloud(np.zeros((0, 5), np.float32), pos) == 0           # "cloud is empty.": unchanged
    assert same_state(before, g.State())
    far = sequence()[1][0].copy()
    far[777, 0] = 2.0e5                                                        # voxel index 2e6 >= 2^20
    with pytest.raises(smb.CheckFailure):
        g.InsertPointCloud(far, (1.0, 0.0, 0.0))
    with pytest.raises(smb.CheckFailure):
        g.InsertPointCloud(sequence()[1][0], (np.nan, 0.0, 0.0))              # the origin too
    assert same_state(before, g.State())
    dirty, pos1 = sequence()[1]
    dirty = dirty.copy()
    dirty[[5, 500, 50_000], [0, 1, 2]] = [np.nan, np.inf, -np.inf]
    assert g.InsertPointCloud(dirty, pos1) == 3 and o.InsertPointCloud(dirty, pos1) == 3
    assert same_state(g.State(), o.State())
    for rgb in (0, 1):
        assert np.array_equal(g.OutputToPointCloud(0.5, rgb).view(np.uint32), o.OutputToPointCloud(0.5, rgb).view(np.uint32))


def test_settings_are_checked():
    for bad in ({"hit_prob": 0.5}, {"miss_prob": 0.5}, {"max_point_num_in_cell": 0}, {"high_resolution": 0.0}):
        with pytest.raises(smb.CheckFailure):
            gpu_map(**bad)
    g = gpu_map()
    g.InsertPointCloud(sequence()[0][0], sequence()[0][1])
    with pytest.raises(smb.CheckFailure):
        g.OutputToPointCloud(1.0)                                             # threshold * 256 outside a uint8


def test_device_insert_equals_host_insert():
    import torch
    a, b = gpu_map(), gpu_map()
    stream = torch.cuda.Stream()
    for pts, pos in sequence()[:4]:
        a.InsertPointCloud(pts, pos)
        with torch.cuda.stream(stream):
            t = torch.from_numpy(pts).cuda(non_blocking=False)
            b.InsertPointCloud(t, pos)
    assert same_state(a.State(), b.State())
    assert np.array_equal(a.OutputToPointCloud(0.6).view(np.uint32), b.OutputToPointCloud(0.6).view(np.uint32))


def test_moving_box_is_removed_walls_and_ground_remain():
    scene = synth.make_scene(seed=3)
    with_box = dict(scene)
    with_box["lo"] = np.vstack([scene["lo"], BOX_LO]); with_box["hi"] = np.vstack([scene["hi"], BOX_HI])
    g = gpu_map()
    o = O.Mrvm()

    def box_points(out):
        return ((out[:, :3] > BOX_LO + [-0.1, -0.1, 0.2]) & (out[:, :3] < BOX_HI + 0.1)).all(axis=1).sum()

    for k in range(10):
        pts, pos = scan(k, with_box if k < 3 else scene, seed_base=100)
        g.InsertPointCloud(pts, pos); o.InsertPointCloud(pts, pos)
        if k == 2:
            assert box_points(g.OutputToPointCloud(0.57)) > 1000          # the parked object is in the map
    out = g.OutputToPointCloud(0.57)
    assert np.array_equal(out.view(np.uint32), o.OutputToPointCloud(0.57).view(np.uint32))
    assert box_points(out) == 0                                            # ... and gone once it has left
    assert (out[:, 2] < -1.6).sum() > 200_000 and (np.abs(out[:, 1]) > 9.8).sum() > 100_000   # ground, walls


def test_cpp_adapter_end_to_end(tmp_path):
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if cxx is None:
        pytest.skip("no g++")
    libdir = os.path.join(ROOT, "staticmapping_b200")
    exe = str(tmp_path / "mrvm_run")
    r = subprocess.run([cxx, "-std=c++14", "-O1", "-Wall", "-I", os.path.join(ROOT, "tests", "stubs"), "-I",
                        os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "adapter"),
                        os.path.join(ROOT, "tests", "cpp", "mrvm_run.cc"), "-o", exe, "-L", libdir, "-l:libsm_b200.so",
                        "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    scans = sequence()[:3]
    with open(tmp_path / "in.bin", "wb") as f:
        f.write(struct.pack("<q", len(scans)))
        for pts, pos in scans:
            f.write(struct.pack("<q", pts.shape[0]))
            f.write(np.asarray(pos, np.float32).tobytes())
            f.write(pts.tobytes())
    r = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    got = np.fromfile(tmp_path / "out.bin", np.float32).reshape(-1, 4)
    o = O.Mrvm(output_average=1)
    for pts, pos in scans:
        o.InsertPointCloud(pts, pos)
    want = o.OutputToPointCloud(0.6, 0)
    assert got.shape == want.shape and np.array_equal(got.view(np.uint32), want.view(np.uint32))
