"""Throughput of the scan pre-processing filter chain (pre_processers::filter::Factory) on the GPU: full-size lidar
scans (synth.lidar_scan, 120 000 points) through three chains:
  default   Range (4.5 - 75 m) + RandomSampler (0.35)            static_mapping_default.xml, lidar_only.xml, lidar_imu*.xml
  kitti     Range + AxisRange + RandomSampler (0.5)              lidar_only_kitti.xml
  ground    Range + RangeImage + GroundRemoval2 + RandomSampler  the kitti config with GroundRemoval2 switched on

Per chain: scans/s from host input (upload included) and from device input (sm_filter_chain_filter_device on a
resident tensor), each a host clock around calls that end in a stream synchronise; the median per-stage device time
from the chain's CUDA events; and the serial oracle (tests/cpp/filters_oracle.cc, one thread) on the host.  Device
name and power limit are read in the same run.

    python profiles/time_filters.py --scans 50 --out profiles/r04_time_filters.json
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

F, I = 1, 0
RANGE = ("Range", {"min_range": (F, "4.5"), "max_range": (F, "75")})
CHAINS = {
    "default": [RANGE, ("RandomSampler", {"sampling_rate": (F, "0.35")})],
    "kitti": [("Range", {"min_range": (F, "5.")}), ("AxisRange", {"min": (F, "-2.")}),
              ("RandomSampler", {"sampling_rate": (F, "0.5")})],
    "ground": [("Range", {"min_range": (F, "5.")}), ("RangeImage", {"top_angle": (F, "3"), "btm_angle": (F, "-25"),
                                                                     "vertical_line_num": (I, "64"),
                                                                     "horizontal_line_num": (I, "1800")}),
               ("GroundRemoval2", {"r_min": (F, "0.1"), "start_ground_height": (F, "-1.5"),
                                   "long_line_threshold": (F, "10"), "max_slope": (F, "0.12"),
                                   "max_error": (F, "0.1"), "max_dist_to_line": (F, "0.10"),
                                   "max_start_height": (F, "0.6")}),
               ("RandomSampler", {"sampling_rate": (F, "0.5")})],
}


def scans(n):
    scene = synth.make_scene(seed=5)
    out = []
    for k in range(n):
        p = synth.lidar_scan(scene, (0.5 * k, 0.0, 0.0), seed=100 + k)
        r = np.zeros((p.shape[0], 5), np.float32)
        r[:, :3] = p
        r[:, 3] = 50.0
        r[:, 4] = np.linspace(0, 1, p.shape[0], dtype=np.float32)
        out.append(r)
    return out


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:
        q = f"nvidia-smi unavailable: {e}"
    return {"device": name, "nvidia_smi": q}


def build(chain, stages):
    for name, params in stages:
        k = chain.add(name)
        assert k >= 0, name
        for pname, (t, text) in params.items():
            assert chain.set_param(k, pname, t, text) == 0, pname
    return chain


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=50)
    ap.add_argument("--oracle-scans", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import filters_oracle as O

    seq = scans(a.scans)
    dev_seq = [torch.from_numpy(p).cuda() for p in seq]
    torch.cuda.synchronize()
    res = {"workload": f"{a.scans} synth.lidar_scan scans x {seq[0].shape[0]} points per chain", **device_info(),
           "chains": {}}
    for label, stages in CHAINS.items():
        g = build(smb.FilterChain(0), stages)
        for p in seq[:3]:                                   # warm-up: module load, workspace allocation
            g.filter(p)
        f = smb.FilterFactory(0, chain=g)
        f.FilterDevice(dev_seq[0])
        torch.cuda.synchronize()
        per_scan, stage_ms, outs = [], [], 0
        t0 = time.perf_counter()
        for p in seq:
            t = time.perf_counter()
            rc, out, _ = g.filter(p)
            per_scan.append(time.perf_counter() - t)
            stage_ms.append(g.stage_ms())
            outs += out.shape[0]
        host_s = time.perf_counter() - t0
        torch.cuda.synchronize()
        dev_scan = []
        t0 = time.perf_counter()
        for t_in in dev_seq:
            t = time.perf_counter()
            f.FilterDevice(t_in)
            dev_scan.append(time.perf_counter() - t)
        dev_s = time.perf_counter() - t0
        o = build(O.Chain(), stages)
        t0 = time.perf_counter()
        for p in seq[:a.oracle_scans]:
            o.filter(p)
        oracle_s = time.perf_counter() - t0
        sm = np.median(np.array(stage_ms), axis=0)
        res["chains"][label] = {
            "stages": [n for n, _ in stages],
            "gpu_host_input_scans_per_s": a.scans / host_s,
            "gpu_host_input_ms_median": 1e3 * float(np.median(per_scan)),
            "gpu_device_input_scans_per_s": a.scans / dev_s,
            "gpu_device_input_ms_median": 1e3 * float(np.median(dev_scan)),
            "stage_device_ms_median_from_cuda_events": {f"{k}:{n}": float(v) for k, (n, v) in
                                                        enumerate(zip([n for n, _ in stages], sm))},
            "mean_output_points": outs / a.scans,
            "oracle_serial_host_scans_per_s": a.oracle_scans / oracle_s,
        }
    res["note"] = ("scan time = host clock around one filter call, which ends in a stream synchronise; host input "
                   "includes the host-to-device copy of the scan and the device-to-host copy of the result; a fused "
                   "run of point-wise stages is reported on its first stage")
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
