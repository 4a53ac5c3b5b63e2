"""TEST INFRASTRUCTURE ONLY — ctypes binding of the loop-closure oracle (oracle/loop_oracle.cpp, built with the VoxelGrid
oracle it reuses into oracle/liblooporacle.so with the flags of oracle/Makefile).  Registration reuses binding.OracleNdt.
PARITY UNPINNED: see oracle/oracle.h and the header of loop_oracle.cpp.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_SRCS = ("loop_oracle.cpp", "voxelgrid_oracle.cpp")


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "liblooporacle.so")
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
        L.orc_loop_detect.restype = None
        L.orc_loop_detect.argtypes = [vp, vp, i64, vp, i64, C.c_float, C.c_double, vp, vp]
        L.orc_loop_submap.restype = i64
        L.orc_loop_submap.argtypes = [vp, vp, vp, i64, i64, i32, C.c_float, vp, vp, vp, vp, i64]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def loop_detect(poses6, times, cur, radius, time_gap):
    """detectLoopClosureDistance for each query keyframe in cur: (pre int64 [Q], -1 = none; squared distance float32 [Q])."""
    poses = np.ascontiguousarray(poses6, dtype=np.float32).reshape(-1, 6)
    t = np.ascontiguousarray(times, dtype=np.float64)
    cur = np.ascontiguousarray(cur, dtype=np.int64).reshape(-1)
    pre = np.empty(len(cur), np.int64)
    d2 = np.empty(len(cur), np.float32)
    lib().orc_loop_detect(_p(poses), _p(t), len(poses), _p(cur), len(cur), radius, time_gap, _p(pre), _p(d2))
    return pre, d2


class Keyframes:
    """The clouds ([n_k, 4] float32, lidar frame) and poses ([K, 6]: x y z roll pitch yaw) of a session, packed once."""

    def __init__(self, clouds, poses6):
        self.off = np.zeros(len(clouds) + 1, np.int64)
        self.off[1:] = np.cumsum([len(c) for c in clouds])
        self.xyzi = np.ascontiguousarray(np.concatenate([np.asarray(c, np.float32).reshape(-1, 4) for c in clouds] + [np.zeros((1, 4), np.float32)]))
        self.poses = np.ascontiguousarray(poses6, dtype=np.float32).reshape(-1, 6)

    def submap(self, key, num, leaf):
        """loopFindNearKeyframes(key, num): (raw concatenation [n, 4], VoxelGrid(leaf) [m, 4], counts [m])."""
        K = len(self.poses)
        lo, hi = max(0, key - num), min(K - 1, key + num)
        n_max = int(self.off[hi + 1] - self.off[lo])
        raw = np.empty((max(n_max, 1), 4), np.float32)
        out = np.empty((max(n_max, 1), 4), np.float32)
        cnt = np.empty(max(n_max, 1), np.int32)
        n_raw = C.c_int64()
        m = lib().orc_loop_submap(_p(self.xyzi), _p(self.off), _p(self.poses), K, key, num, leaf, _p(raw), C.byref(n_raw), _p(out), _p(cnt), n_max)
        return raw[: n_raw.value].copy(), out[:m].copy(), cnt[:m].copy()
