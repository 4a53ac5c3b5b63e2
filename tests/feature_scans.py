"""Scans for the LOAM front-end tests (oracle self-check and device parity): small constructed scans that reach every quirk of
the contract in oracle/feature_oracle.cpp, as (records, stride, intensity offset, ring offset, ring bytes, FeatureParams)."""
import math

import numpy as np

from oracle.feature_binding import FeatureParams, records

F = np.float32


def spinning(n_scan=16, H=360, seed=0, dup=0.0, junk=0.0, rate=1):
    """A spinning-lidar scan of boxes and walls: occlusions, steps, planes; dup = fraction of second returns, junk = fraction of
    non-finite / out-of-range points and bad rings."""
    rng = np.random.default_rng(seed)
    xyz, ring = [], []
    for r in range(n_scan):
        el = math.radians(-15.0 + 30.0 * r / max(n_scan - 1, 1))
        for c in range(H):
            if rng.random() < 0.03 or (r % 4 == 1 and 100 <= c < 100 + H // 12):  # drop-outs and a wide gap
                continue
            az = 2 * math.pi * c / H
            d = 8.0 + 4.0 * math.sin(3 * az) + (5.0 if (c // 37) % 3 == 0 else 0.0) + rng.normal(0, 0.01)
            if rng.random() < 0.05:
                d *= 0.5
            xyz.append((d * math.cos(el) * math.cos(az), d * math.cos(el) * math.sin(az), d * math.sin(el)))
            ring.append(r)
    xyz, ring = np.array(xyz, F), np.array(ring, np.int64)
    if dup:
        k = rng.random(len(xyz)) < dup
        xyz = np.concatenate([xyz, xyz[k] * F(1.01)])
        ring = np.concatenate([ring, ring[k]])
        p = rng.permutation(len(xyz))
        xyz, ring = xyz[p], ring[p]
    if junk:
        k = np.flatnonzero(rng.random(len(xyz)) < junk)
        kinds = rng.integers(0, 5, len(k))
        xyz[k[kinds == 0], 0] = np.nan
        xyz[k[kinds == 1], 2] = np.inf
        xyz[k[kinds == 2]] *= F(1e-3)  # inside lidarMinRange
        xyz[k[kinds == 3]] *= F(2e3)   # beyond lidarMaxRange
        ring[k[kinds == 4]] = n_scan + 3
    inten = (np.arange(len(xyz)) % 97).astype(F)
    return (*records(xyz, inten, ring), FeatureParams(n_scan=n_scan, horizon_scan=H, downsample_rate=rate))


def livox(n_lines=6, per_line=400, H=300, seed=1):
    """A Livox-shaped scan (petal pattern, points in arrival order, lines interleaved) whose lines carry more points than
    Horizon_SCAN, so the per-line counters run past it."""
    rng = np.random.default_rng(seed)
    t = np.arange(n_lines * per_line)
    line = (t % n_lines).astype(np.uint8)
    th = t * 0.013
    rad = np.abs(np.sin(2.5 * th)) * 0.6
    d = 10.0 + 3.0 * (np.floor(th * 2) % 2) + rng.normal(0, 0.02, len(t))
    xyz = np.stack([d, d * rad * np.cos(th), d * rad * np.sin(th)], 1).astype(F)
    return (*records(xyz, (t % 31).astype(F), line, np.uint8), FeatureParams(n_scan=n_lines, horizon_scan=H, sensor=1))


def quirks(H=1800):
    """Livox-mode rings (columns = arrival order, ranges exact: every point lies on the x axis) built to reach the quirks:
    two leading empty rings, a ring of 7 points, a ring of equal ranges (curvature ties at zero), rings of periodic steps and
    V-shaped dents (equal curvatures above edgeThreshold, more than 20 corner candidates per region), a ring longer than
    Horizon_SCAN, and a stepped ring (occlusion marks)."""
    ranges, ring = [], []

    def add(r, rr):
        ranges.extend(rr)
        ring.extend([r] * len(rr))

    add(2, [9.0] * 200)
    add(3, [7.0] * 7)
    add(4, [10.0 + (3.0 if c % 4 == 0 else 0.0) for c in range(H)])
    add(5, [12.0 + 0.1 * abs(c % 12 - 6) for c in range(H)])  # V-shaped: equal curvatures of 9, not parallel-beam marked
    add(6, [6.0 + 0.25 * (c % 9) for c in range(H + 40)])
    add(7, [5.0 + (2.0 if (c // 15) % 2 else 0.0) for c in range(H)])
    r = np.array(ranges, F)
    xyz = np.stack([r, np.zeros_like(r), np.zeros_like(r)], 1)
    return (*records(xyz, np.arange(len(xyz)).astype(F), np.array(ring), np.uint8), FeatureParams(n_scan=8, horizon_scan=H, sensor=1))
