"""Seeded input builders shared by the parity tests (SURVEY.md section 8d)."""
from __future__ import annotations

import functools

import numpy as np

from staticmapping_b200 import synth


def se3_error(A, B):
    """(translation error [m], rotation angle [rad]) between two 4x4 transforms.  The angle is
    atan2(sin, cos) of the relative rotation: arccos of the trace alone cannot resolve angles below
    2.1e-8 rad, the angle it returns when the trace is one rounding step below 3."""
    E = np.linalg.inv(A) @ B
    R = E[:3, :3]
    s = 0.5 * np.linalg.norm([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    c = 0.5 * (np.trace(R) - 1.0)
    return float(np.linalg.norm(E[:3, 3])), float(np.arctan2(s, c))


@functools.lru_cache(maxsize=None)
def corner_pair():
    """Config 1: two 5k clouds of the 3-plane corner; returns (source f64, target raw f64, GT)."""
    tgt = synth.corner_scene_cloud(5000, 1234).astype(np.float64)
    GT = synth.corner_ground_truth()
    scene2 = synth.corner_scene_cloud(5000, 5678).astype(np.float64)
    src = synth.apply_se3(np.linalg.inv(GT), scene2).astype(np.float32).astype(np.float64)
    return src, tgt, GT


@functools.lru_cache(maxsize=None)
def lidar_pair(n_az=300, n_beams=32, submap_points=60000, pair=0, seed=0):
    """Reduced-size config-2 analogue: scan -> submap of the synthetic street scene.
    Returns (source f64 (Ns,3), target raw f64 (Nt,3), perturbation 4x4)."""
    scene = synth.make_scene(seed)
    sub = synth.submap(scene, seed=seed, n_points=submap_points, n_scans=5, n_beams=n_beams,
                       n_az=n_az).astype(np.float64)
    scan = synth.lidar_scan(scene, (2.0, 0.0, 0.0), seed=seed * 131 + 77 + pair, n_beams=n_beams,
                            n_az=n_az).astype(np.float64)
    world = scan + np.array([2.0, 0.0, 0.0])
    P = synth.perturbation(pair)
    src = synth.apply_se3(np.linalg.inv(P), world).astype(np.float32).astype(np.float64)
    return src, sub, P


def full_size_pair(pair=0):
    """BASELINE.json configs[1]/[2]/[4] sizes: one 64-beam x 1875-azimuth scan (120 000 points)
    against a 500 000-point submap (SURVEY.md section 8d)."""
    src, sub, P = lidar_pair(n_az=1875, n_beams=64, submap_points=500_000, pair=pair)
    assert src.shape == (120_000, 3) and sub.shape == (500_000, 3)
    return src, sub, P


def reference_voxel_test_cloud():
    """The cloud of the reference's own unit test (pre_processors/test/test_filter_voxel_grid.cc:54-63):
    a 10 x 10 lattice, x = i*0.1f + 0.02f, y = j*0.1f + 0.02f, z = 0.1f, intensity 0 (float arithmetic)."""
    pts = np.zeros((100, 5), np.float32)
    k = 0
    for x in range(10):
        for y in range(10):
            pts[k, 0] = np.float32(x) * np.float32(0.1) + np.float32(0.02)
            pts[k, 1] = np.float32(y) * np.float32(0.1) + np.float32(0.02)
            pts[k, 2] = np.float32(0.1)
            k += 1
    return pts
