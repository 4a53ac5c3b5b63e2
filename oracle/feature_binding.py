"""TEST INFRASTRUCTURE ONLY — ctypes binding of the LOAM front-end oracle (oracle/feature_oracle.cpp, built with the VoxelGrid
oracle it reuses into oracle/libfeatureoracle.so with the flags of oracle/Makefile).
PARITY UNPINNED: see oracle/oracle.h and the header of feature_oracle.cpp.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_SRCS = ("feature_oracle.cpp", "voxelgrid_oracle.cpp")


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "libfeatureoracle.so")
    deps = [os.path.join(_HERE, f) for f in _SRCS + ("oracle.h",)]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in deps):
        subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O3", "-fopenmp", "-ffp-contract=off", "-fPIC", "-Wall", "-shared", "-o", so]
                              + [os.path.join(_HERE, f) for f in _SRCS])
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
        L.orc_features.restype = i64
        L.orc_features.argtypes = [vp, i64, i64, i64, i64, i32, vp, vp] + [vp] * 13
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@dataclass
class FeatureParams:
    """LIO-SAM's parameters with its defaults; sensor 0 = velodyne / ouster (column from the azimuth), 1 = livox."""
    n_scan: int = 16
    horizon_scan: int = 1800
    downsample_rate: int = 1
    sensor: int = 0
    min_range: float = 1.0
    max_range: float = 1000.0
    edge_threshold: float = 1.0
    surf_threshold: float = 0.1
    odometry_surf_leaf: float = 0.4
    mapping_corner_leaf: float = 0.2
    mapping_surf_leaf: float = 0.4


COUNT_NAMES = ("dropped_nonfinite", "dropped_range", "dropped_row", "dropped_col", "dropped_dup", "n_extracted", "n_corner", "n_surface",
               "n_corner_ds", "n_surf_ds")


def records(xyz, intensity=None, ring=None, ring_dtype=np.uint16):
    """Packs a scan as PointXYZIR-like records: x y z intensity (float32) ring (ring_dtype) padded to 24 bytes.
    Returns (bytes array [n, 24] uint8, stride, intensity offset, ring offset, ring bytes)."""
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    n = len(xyz)
    rec = np.zeros((n, 24), np.uint8)
    rec[:, 0:12] = xyz.view(np.uint8).reshape(n, 12)
    rec[:, 12:16] = np.asarray(intensity if intensity is not None else np.zeros(n), np.float32).reshape(n, 1).view(np.uint8)
    rb = np.dtype(ring_dtype).itemsize
    rec[:, 16:16 + rb] = np.asarray(ring if ring is not None else np.zeros(n), ring_dtype).reshape(n, 1).view(np.uint8)
    return rec, 24, 12, 16, rb


def features(rec, stride, int_off, ring_off, ring_bytes, prm: FeatureParams):
    """Steps 1-6 of the contract on one scan: a dict of every intermediate (see orc_features)."""
    rec = np.ascontiguousarray(rec, dtype=np.uint8)
    n = rec.size // stride
    cap = max(n, 1)
    iprm = np.array([prm.n_scan, prm.horizon_scan, prm.downsample_rate, prm.sensor], np.int32)
    fprm = np.array([prm.min_range, prm.max_range, prm.edge_threshold, prm.surf_threshold, prm.odometry_surf_leaf, prm.mapping_corner_leaf,
                     prm.mapping_surf_leaf], np.float32)
    cloud = np.empty((cap, 4), np.float32)
    col, rng = np.empty(cap, np.int32), np.empty(cap, np.float32)
    start, end = np.empty(prm.n_scan, np.int32), np.empty(prm.n_scan, np.int32)
    curv, label, picked = np.empty(cap, np.float32), np.empty(cap, np.int8), np.empty(cap, np.uint8)
    clouds = [np.empty((cap, 4), np.float32) for _ in range(4)]
    counts = np.zeros(10, np.int64)
    lib().orc_features(_p(rec), n, stride, int_off, ring_off, ring_bytes, _p(iprm), _p(fprm), _p(cloud), _p(col), _p(rng), _p(start), _p(end),
                       _p(curv), _p(label), _p(picked), *[_p(c) for c in clouds], _p(counts))
    m = int(counts[5])
    out = dict(zip(COUNT_NAMES, (int(c) for c in counts)))
    out.update(cloud=cloud[:m].copy(), col=col[:m].copy(), range=rng[:m].copy(), start=start, end=end, curvature=curv[:m].copy(),
               label=label[:m].copy(), picked=picked[:m].copy())
    for name, c, k in zip(("corner", "surface", "corner_ds", "surf_ds"), clouds, counts[6:10]):
        out[name] = c[: int(k)].copy()
    return out
