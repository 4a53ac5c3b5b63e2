"""TEST INFRASTRUCTURE ONLY — ctypes binding of the LOAM local-map oracle (oracle/surround_oracle.cpp, built with the VoxelGrid
oracle it reuses into oracle/libsurroundoracle.so with the flags of oracle/Makefile).
PARITY UNPINNED: see oracle/oracle.h and the header of surround_oracle.cpp.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_SRCS = ("surround_oracle.cpp", "voxelgrid_oracle.cpp")


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "libsurroundoracle.so")
    deps = [os.path.join(_HERE, f) for f in _SRCS + ("oracle.h",)]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in deps):
        subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O3", "-fopenmp", "-ffp-contract=off", "-fPIC", "-Wall", "-shared", "-o", so]
                              + [os.path.join(_HERE, f) for f in _SRCS])
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        vp, i64 = C.c_void_p, C.c_int64
        L.orc_loam_surrounding.restype = None
        L.orc_loam_surrounding.argtypes = [vp, vp, vp, vp, vp, i64, C.c_double, vp, vp, vp, vp, vp, vp, vp, vp, i64]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Keyframes:
    """The clouds ([n_k, 4] float32, lidar frame), poses ([K, 6]: x y z roll pitch yaw) and times (s) of a session, packed once.
    The first n_corner[k] points of cloud k are its corner cloud, the rest its surf cloud."""

    def __init__(self, clouds, poses6, times, n_corner):
        self.off = np.zeros(len(clouds) + 1, np.int64)
        self.off[1:] = np.cumsum([len(c) for c in clouds])
        self.xyzi = np.ascontiguousarray(np.concatenate([np.asarray(c, np.float32).reshape(-1, 4) for c in clouds] + [np.zeros((1, 4), np.float32)]))
        self.poses = np.ascontiguousarray(poses6, dtype=np.float32).reshape(-1, 6)
        self.times = np.ascontiguousarray(times, dtype=np.float64)
        self.n_corner = np.ascontiguousarray(n_corner, dtype=np.int64)

    def surrounding(self, cur, time_cur, search_radius=50.0, density=2.0, corner_leaf=0.2, surf_leaf=0.4):
        """extractSurroundingKeyFrames with keyframe cur the newest (-1: the last): (keys after the distance gate int64, list
        length before the gate, laserCloudCornerFromMapDS [m, 4], laserCloudSurfFromMapDS [m, 4])."""
        cur = len(self.poses) - 1 if cur < 0 else cur
        prm = np.array([search_radius, density, corner_leaf, surf_leaf], np.float32)
        keys = np.empty(2 * (cur + 1), np.int64)
        cap = max(int(self.off[-1]) * 2, 1)
        co, so = np.empty((cap, 4), np.float32), np.empty((cap, 4), np.float32)
        nk, nl, nc, ns = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
        lib().orc_loam_surrounding(_p(self.xyzi), _p(self.off), _p(self.n_corner), _p(self.poses), _p(self.times), cur, time_cur, _p(prm), _p(keys),
                                   C.byref(nk), C.byref(nl), _p(co), C.byref(nc), _p(so), C.byref(ns), cap)
        return keys[: nk.value].copy(), nl.value, co[: nc.value].copy(), so[: ns.value].copy()
