"""Throughput of MultiResolutionVoxelMap on the GPU: a sequence of full-size lidar scans (synth.lidar_scan, 120 000
points, the sensor moving 1 m per scan) inserted at 0.1 m, then one OutputToPointCloud.

Reports scans/s and ray-voxel visits/s (visits counted here: every voxel of every Bresenham ray, max |delta| + 1 per
point, the walk the reference does per point), the device time of each insert phase from the map's CUDA events, the
output time, and the serial oracle on the host (a one-thread restatement, not the reference's 10-thread OpenMP loop)
over the first --oracle-scans scans.  Device name and power limit are read in the same run.

    python profiles/time_mrvm.py --scans 50 --out profiles/r03_time_mrvm.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import staticmapping_b200 as smb  # noqa: E402
from staticmapping_b200 import synth  # noqa: E402


def scans(n, step):
    scene = synth.make_scene(seed=3)
    out = []
    for k in range(n):
        pos = np.array([float(k), 0.0, 0.0])
        p = synth.lidar_scan(scene, pos, seed=k)
        pts = np.zeros((p.shape[0], 5), np.float32)
        pts[:, :3] = p + pos.astype(np.float32)
        pts[:, 3] = np.random.default_rng(k).uniform(0, 180, p.shape[0]).astype(np.float32)
        o = np.floor(pos.astype(np.float32) / np.float32(step))
        e = np.floor(pts[:, :3] / np.float32(step))
        visits = int((np.abs(e - o).max(axis=1) + 1).sum())
        out.append((pts, pos, visits))
    return out


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:        # the number still stands with the torch device name
        q = f"nvidia-smi unavailable: {e}"
    return {"device": name, "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=50)
    ap.add_argument("--oracle-scans", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU")
    step = 0.1
    t = time.perf_counter()
    seq = scans(a.scans, step)
    gen_s = time.perf_counter() - t
    settings = smb.MrvmSettings(high_resolution=step)

    warm = smb.MultiResolutionVoxelMap()
    warm.Initialise(settings)
    for pts, pos, _ in seq[:3]:
        warm.InsertPointCloud(pts, pos)
    warm.OutputToPointCloud(0.6)
    del warm

    m = smb.MultiResolutionVoxelMap(expected_voxels=1 << 22)
    m.Initialise(settings)
    per_scan = []
    t0 = time.perf_counter()
    for pts, pos, _ in seq:
        t = time.perf_counter()
        m.InsertPointCloud(pts, pos)                 # returns after the device work has finished
        per_scan.append(time.perf_counter() - t)
    insert_s = time.perf_counter() - t0
    t = time.perf_counter()
    out = m.OutputToPointCloud(0.6)
    output_s = time.perf_counter() - t
    phases = m.PhaseMs()
    visits = sum(v for _, _, v in seq)

    import mrvm_oracle as O
    o = O.Mrvm(high_resolution=step)
    t = time.perf_counter()
    for pts, pos, _ in seq[:a.oracle_scans]:
        o.InsertPointCloud(pts, pos)
    oracle_s = time.perf_counter() - t
    oracle_visits = sum(v for _, _, v in seq[:a.oracle_scans])

    res = {
        "workload": f"{a.scans} synth.lidar_scan scans x {seq[0][0].shape[0]} points, sensor +1 m per scan, "
                    f"high_resolution {step} m, then OutputToPointCloud(0.6)",
        **device_info(),
        "gpu": {
            "scans_per_s": a.scans / insert_s,
            "ray_voxel_visits": visits,
            "ray_voxel_visits_per_s": visits / insert_s,
            "insert_ms_mean": 1e3 * insert_s / a.scans,
            "insert_ms_median": 1e3 * float(np.median(per_scan)),
            "insert_ms_last10_mean": 1e3 * float(np.mean(per_scan[-10:])),
            "phase_ms_total_from_cuda_events": {k: v for k, v in phases.items() if k != "inserts"},
            "output_ms": 1e3 * output_s,
            "voxels": m.size(),
            "output_points": int(out.shape[0]),
            "note": "insert time = host clock around each insert, which ends in a stream synchronise; includes the "
                    "host-to-device copy of the scan (upload phase)",
        },
        "oracle_serial_host": {
            "label": "one-thread C++ restatement (tests/cpp/mrvm_oracle.cc) on the host CPU, not the reference's "
                     "10-thread OpenMP loop",
            "scans": a.oracle_scans,
            "scans_per_s": a.oracle_scans / oracle_s,
            "ray_voxel_visits_per_s": oracle_visits / oracle_s,
        },
        "scan_generation_s": gen_s,
    }
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
