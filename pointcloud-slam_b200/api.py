"""ctypes view of the b200reg C ABI (include/b200reg.h) with the reference's interface names.

This is the Python mirror used by tests/ and bench.py; the C++ mirror a ROS package would compile
lives in host/*.hpp.  Class and method names follow the reference:
  IVox.AddPoints / GetClosestPoint / NumValidGrids              (jueying_lio ivox3d.h:53-88)
  Esekf.update_iterated_dyn_share_modified / get_x / get_P      (IKFoM esekfom.hpp:1526,1836-1848)
  LaserMappingCore.MapIncremental                               (jueying_lio laser_mapping.cc:525)
  NormalDistributionsTransform.setInputTarget / align / ...     (pclomp ndt_omp.h:117-261)
There is no CPU fallback: if libb200reg.so is missing or no CUDA device exists, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
B200_MAX_PASSES = 8


class B200Error(RuntimeError):
    pass


class MapParams(C.Structure):
    _fields_ = [("resolution", C.c_float), ("nearby", C.c_int32), ("capacity_voxels", C.c_uint64),
                ("max_range", C.c_float), ("max_points", C.c_uint64)]


class IekfParams(C.Structure):
    _fields_ = [("max_iter", C.c_int32), ("plane_thr", C.c_float), ("extrinsic_est_en", C.c_int32), ("R", C.c_double),
                ("limit", C.c_double * 23), ("filter_size_map", C.c_double)]


class IekfStats(C.Structure):
    _fields_ = [("status", C.c_int32), ("passes", C.c_int32), ("knn_passes", C.c_int32), ("converged", C.c_int32),
                ("n_eff", C.c_int32 * B200_MAX_PASSES), ("knn", C.c_int32 * B200_MAX_PASSES), ("gpu_ms", C.c_float)]


class NdtParams(C.Structure):
    _fields_ = [("resolution", C.c_float), ("step_size", C.c_double), ("outlier_ratio", C.c_double),
                ("trans_eps", C.c_double), ("max_iter", C.c_int32), ("search", C.c_int32), ("min_pts", C.c_int32),
                ("eig_ratio", C.c_double)]


class NdtResult(C.Structure):
    _fields_ = [("converged", C.c_int32), ("iters", C.c_int32), ("evals", C.c_int32), ("hess_evals", C.c_int32),
                ("trans_probability", C.c_double), ("hessian", C.c_double * 36), ("score", C.c_double),
                ("p_final", C.c_double * 6), ("gpu_ms", C.c_float)]


class NdtPairResult(C.Structure):
    """b200_ndt_pair_result (include/b200reg.h)."""
    _fields_ = [("status", C.c_int32), ("ndt", NdtResult), ("fitness", C.c_double), ("n_in_range", C.c_int64),
                ("final16", C.c_float * 16)]


class GicpParams(C.Structure):
    _fields_ = [("k_correspondences", C.c_int32), ("gicp_epsilon", C.c_double), ("rotation_epsilon", C.c_double),
                ("transformation_epsilon", C.c_double), ("corr_dist_threshold", C.c_double), ("max_iterations", C.c_int32),
                ("max_inner_iterations", C.c_int32)]


class GicpResult(C.Structure):
    _fields_ = [("converged", C.c_int32), ("iterations", C.c_int32), ("last_m", C.c_int32), ("last_inner", C.c_int32),
                ("last_status", C.c_int32), ("inner_total", C.c_int32), ("n_f", C.c_int32), ("n_df", C.c_int32), ("n_fdf", C.c_int32),
                ("delta", C.c_double), ("gpu_ms", C.c_float)]


class LoamStats(C.Structure):
    _fields_ = [("iters", C.c_int32), ("n_sel", C.c_int32), ("converged", C.c_int32), ("degenerate", C.c_int32), ("gpu_ms", C.c_float),
                ("AtA_first", C.c_double * 36)]


def lib_path() -> str:
    # B200REG_LIB: development override for A/B timing of two builds of the SAME engine (never a different implementation)
    return os.environ.get("B200REG_LIB") or os.path.join(_HERE, "libb200reg.so")


def build(verbose: bool = False) -> str:
    """Compile libb200reg.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "-j8"]
    if not verbose:
        cmd.append("-s")
    subprocess.check_call(cmd)
    return lib_path()


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise B200Error(f"{path} is missing: run __graft_entry__.build() (there is no CPU fallback)")
    L = C.CDLL(path)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
    L.b200_version.restype = C.c_char_p
    L.b200_last_error.restype = C.c_char_p
    L.b200_kernel_launches.restype = i64
    L.b200_map_create.argtypes = [C.POINTER(MapParams), i32, C.POINTER(vp)]
    L.b200_map_destroy.argtypes = [vp]
    L.b200_map_insert.argtypes = [vp, vp, i64, i64]
    L.b200_map_knn5.argtypes = [vp, vp, i64, i64, vp, vp, vp]
    L.b200_map_knn5_points.argtypes = [vp, vp, i64, i64, vp, vp, vp, vp]
    L.b200_map_num_voxels.restype = i64
    L.b200_map_num_voxels.argtypes = [vp]
    L.b200_map_num_points.restype = i64
    L.b200_map_num_points.argtypes = [vp]
    L.b200_iekf_create.argtypes = [C.POINTER(IekfParams), vp, C.POINTER(vp)]
    L.b200_iekf_destroy.argtypes = [vp]
    L.b200_iekf_update.argtypes = [vp, vp, i64, i64, vp, vp, C.POINTER(IekfStats)]
    L.b200_iekf_update_device.argtypes = [vp, vp, i64, vp, vp, C.POINTER(IekfStats)]
    L.b200_iekf_last_HtH.argtypes = [vp, i32, vp, vp, vp]
    L.b200_iekf_obs_model.argtypes = [vp, vp, i64, i64, vp, i32, vp, vp, vp]
    L.b200_iekf_point_state.argtypes = [vp, i64, vp, vp, vp, vp, vp]
    L.b200_iekf_map_incremental.argtypes = [vp, vp, i32, vp, vp]
    L.b200_iekf_predict.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    L.b200_iekf_world_scan.argtypes = [vp, vp, vp, i64, i64, vp]
    L.b200_iekf_set_profiling.argtypes = [vp, i32]
    L.b200_iekf_set_graph.argtypes = [vp, i32]
    L.b200_iekf_kernel_times.argtypes = [vp, vp, i32]
    L.b200_iekf_io_bytes.argtypes = [vp, i64, vp, vp]
    L.b200_iekf_launch_modes.argtypes = [vp, vp, vp, vp]
    L.b200_map_stencil_points.argtypes = [vp, vp, i64, i64, vp, vp]
    L.b200_map_last_knn_ms.restype = C.c_float
    L.b200_map_last_knn_ms.argtypes = [vp]
    L.b200_map_tma_timeouts.restype = i64
    L.b200_map_evicted.restype = i64
    L.b200_map_evicted.argtypes = [vp]
    L.b200_map_dropped.restype = i64
    L.b200_map_dropped.argtypes = [vp, vp]
    L.b200_flush_l2.argtypes = [i32]
    L.b200_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.b200_host_free.argtypes = [vp]
    if hasattr(L, "b200_ndt_create"):
        L.b200_ndt_create.argtypes = [C.POINTER(NdtParams), i32, C.POINTER(vp)]
        L.b200_ndt_destroy.argtypes = [vp]
        L.b200_ndt_set_target.argtypes = [vp, vp, i64, i64]
        L.b200_ndt_set_source.argtypes = [vp, vp, i64, i64]
        L.b200_ndt_num_voxels.restype = i64
        L.b200_ndt_num_voxels.argtypes = [vp]
        L.b200_ndt_leaves.restype = i64
        L.b200_ndt_leaves.argtypes = [vp, i64, vp, vp, vp, vp, vp]
        L.b200_ndt_align.argtypes = [vp, vp, vp, C.POINTER(NdtResult)]
        L.b200_ndt_derivatives.argtypes = [vp, vp, vp, vp, vp]
        L.b200_ndt_hessian.argtypes = [vp, vp, vp]
        L.b200_ndt_newton_direction.argtypes = [vp, vp, vp, i32, vp, vp]
        L.b200_ndt_max_eigen.argtypes = [vp, vp]
        L.b200_ndt_score_batch.argtypes = [vp, vp, i64, vp]
        L.b200_comm_unique_id.argtypes = [vp]
        L.b200_comm_init_rank.argtypes = [i32, i32, vp, i32, C.POINTER(vp)]
        L.b200_comm_destroy.argtypes = [vp]
        L.b200_reloc_argmin.argtypes = [vp, vp, vp, i64, i64, vp, vp, vp]
        L.b200_reloc_argmin_strided.argtypes = [vp, vp, vp, i64, i64, i64, vp, vp, vp]
        L.b200_ndt_align_batch.argtypes = [vp, vp, i64, vp, vp]
        L.b200_ndt_grid.argtypes = [vp, vp, vp]
        L.b200_ndt_set_target_bcast.argtypes = [vp, vp, vp, i64, i64, i32]
        L.b200_ndt_nbhd_total.restype = i64
        L.b200_ndt_nbhd_total.argtypes = [vp, vp]
        L.b200_ndt_last_ms.restype = C.c_float
        L.b200_ndt_last_ms.argtypes = [vp]
        L.b200_ndt_last_launches.argtypes = [vp]
        L.b200_ndt_fitness_score.argtypes = [vp, vp, C.c_double, vp, vp]
        L.b200_ndt_last_score_kernel_ms.restype = C.c_float
        L.b200_ndt_last_score_kernel_ms.argtypes = [vp]
        L.b200_ndt_score_pairs.argtypes = [vp, vp, i64, vp]
        L.b200_ndt_stream_barrier.argtypes = [vp, vp]
    if hasattr(L, "b200_ndt_pairs_create"):  # absent from builds older than the batched pair registration (B200REG_LIB A/B timing)
        L.b200_ndt_pairs_create.argtypes = [C.POINTER(NdtParams), i32, C.POINTER(vp)]
        L.b200_ndt_pairs_destroy.argtypes = [vp]
        L.b200_ndt_pairs_align.argtypes = [vp, vp, vp, vp, vp, vp, i64, i64, vp, C.c_double, vp]
        L.b200_ndt_pairs_leaves.restype = i64
        L.b200_ndt_pairs_leaves.argtypes = [vp, i64, i64, vp, vp, vp, vp, vp]
    L.b200_downsampler_create.argtypes = [i32, C.POINTER(vp)]
    L.b200_downsampler_destroy.argtypes = [vp]
    L.b200_voxel_downsample.argtypes = [vp, vp, i64, i64, C.c_float, i32, vp, vp, i64, vp]
    L.b200_scan_undistort.argtypes = [vp, vp, i64, i64, i32, i32, vp, i32, vp, vp, vp]
    L.b200_voxel_downsample_staged.argtypes = [vp, C.c_float, i32, vp]
    L.b200_downsampler_device_points.restype = vp
    L.b200_downsampler_device_points.argtypes = [vp, vp]
    L.b200_downsampler_last_ms.restype = C.c_float
    L.b200_downsampler_last_ms.argtypes = [vp]
    L.b200_mapbuild_create.argtypes = [C.c_float, C.c_uint64, i32, C.POINTER(vp)]
    L.b200_mapbuild_destroy.argtypes = [vp]
    L.b200_mapbuild_add_keyframe.argtypes = [vp, vp, i64, i64, vp]
    L.b200_mapbuild_add_keyframe_device.argtypes = [vp, vp, i64, vp]
    L.b200_mapbuild_add_keyframes_device.argtypes = [vp, vp, vp, vp, i64]
    L.b200_mapbuild_num_voxels.restype = i64
    L.b200_mapbuild_num_voxels.argtypes = [vp]
    L.b200_mapbuild_merge.argtypes = [vp, vp]
    L.b200_mapbuild_extract.restype = i64
    L.b200_mapbuild_extract.argtypes = [vp, vp, vp, i64]
    L.b200_mapbuild_last_exchange_ms.restype = C.c_float
    L.b200_mapbuild_last_exchange_ms.argtypes = [vp]
    L.b200_loam_create.argtypes = [i64, i32, C.POINTER(vp)]
    L.b200_loam_destroy.argtypes = [vp]
    L.b200_loam_set_map.argtypes = [vp, vp, i64, i64, vp, i64, i64]
    L.b200_loam_optimize.argtypes = [vp, vp, i64, i64, vp, i64, i64, vp, i32, C.POINTER(LoamStats)]
    L.b200_loam_features.argtypes = [vp, vp, i64, i64, vp, i64, i64, vp, vp, vp, vp]
    L.b200_gicp_create.argtypes = [C.POINTER(GicpParams), i32, C.POINTER(vp)]
    L.b200_gicp_destroy.argtypes = [vp]
    L.b200_gicp_set_target.argtypes = [vp, vp, i64, i64]
    L.b200_gicp_set_source.argtypes = [vp, vp, i64, i64]
    L.b200_gicp_align.argtypes = [vp, vp, vp, C.POINTER(GicpResult)]
    L.b200_gicp_fitness_score.argtypes = [vp, vp, C.c_double, vp, vp]
    L.b200_gicp_covariances.argtypes = [vp, i32, vp, vp]
    L.b200_gicp_correspondences.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.b200_gicp_cost.argtypes = [vp, vp, vp, vp, vp, vp]
    L.b200_gicp_index_info.argtypes = [vp, i32, vp, vp, vp]
    _LIB = L
    return L


def knn_tma_timeouts() -> int:
    """Queries of the TMA-staged search (B200_KNN_MODE=9) whose bulk copies hit the watchdog and took the gather path (expected 0)."""
    return int(lib().b200_map_tma_timeouts())


def _check(rc: int, soft=(0,)):
    """Negative codes are errors; positive codes are the reference's soft outcomes and are returned."""
    if rc < 0:
        raise B200Error(f"b200reg error {rc}: {lib().b200_last_error().decode()}")
    return rc


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _cloud(a):
    a = np.asarray(a)
    if a.dtype != np.float32 or a.ndim != 2 or a.shape[1] < 3 or a.strides[1] != 4:
        a = np.ascontiguousarray(a, dtype=np.float32)
    return a


class PinnedCloud:
    """A page-locked host array (b200_host_alloc) shaped like a point cloud: scans written into `.array` reach the device
    without the host-side packing pass (include/b200reg.h).  Keep the object alive while the array is in use."""

    def __init__(self, n, cols=3):
        self.ptr = C.c_void_p()
        self.nbytes = int(n) * int(cols) * 4
        _check(lib().b200_host_alloc(C.c_size_t(self.nbytes), C.byref(self.ptr)))
        buf = (C.c_float * (int(n) * int(cols))).from_address(self.ptr.value)
        self.array = np.frombuffer(buf, dtype=np.float32).reshape(int(n), int(cols))

    def close(self):
        if getattr(self, "ptr", None) and self.ptr.value:
            self.array = None
            try:
                lib().b200_host_free(self.ptr)
            except Exception:  # interpreter shutdown: module globals may already be torn down
                pass
            self.ptr = C.c_void_p()

    __del__ = close


def flush_l2(device=0):
    _check(lib().b200_flush_l2(device))


def kernel_launches() -> int:
    return int(lib().b200_kernel_launches())


class IVox:
    """GPU local map with jueying_lio::IVox's surface (ivox3d.h:53-88)."""

    def __init__(self, resolution=0.2, nearby=6, capacity=1_000_000, device=0, max_points=0, max_range=5.0):
        self.params = MapParams(resolution, nearby, capacity, max_range, max_points)
        self.h = C.c_void_p()
        _check(lib().b200_map_create(C.byref(self.params), device, C.byref(self.h)))

    def close(self):
        if getattr(self, "h", None):
            try:
                lib().b200_map_destroy(self.h)
            except TypeError:  # interpreter shutdown: module globals are already torn down
                pass
            self.h = None

    __del__ = close

    def AddPoints(self, points):
        pts = _cloud(points)
        _check(lib().b200_map_insert(self.h, _p(pts), pts.shape[0], pts.strides[0]))

    def GetClosestPoint(self, points):
        """Batched GetClosestPoint(pt, out, 5, 5.0): returns (ordinals [n,5], sqdist [n,5], count [n])."""
        q = _cloud(points)
        n = q.shape[0]
        idx = np.empty((n, 5), np.int32)
        d2 = np.empty((n, 5), np.float32)
        cnt = np.empty(n, np.int32)
        _check(lib().b200_map_knn5(self.h, _p(q), n, q.strides[0], _p(idx), _p(d2), _p(cnt)))
        return idx, d2, cnt

    def GetClosestPointsXYZ(self, points):
        """b200_map_knn5_points: like GetClosestPoint, plus the neighbours' coordinates [n, 5, 3] straight from the device map."""
        q = _cloud(points)
        n = q.shape[0]
        idx = np.empty((n, 5), np.int32)
        d2 = np.empty((n, 5), np.float32)
        cnt = np.empty(n, np.int32)
        nb = np.zeros((n, 5, 3), np.float32)
        _check(lib().b200_map_knn5_points(self.h, _p(q), n, q.strides[0], _p(idx), _p(d2), _p(cnt), _p(nb)))
        return idx, d2, cnt, nb

    def stencil_points(self, points):
        """(sum of map points, occupied cells) over the stencils of the queries — roofline bookkeeping."""
        q = _cloud(points)
        a, b = C.c_int64(0), C.c_int64(0)
        _check(lib().b200_map_stencil_points(self.h, _p(q), q.shape[0], q.strides[0], C.byref(a), C.byref(b)))
        return a.value, b.value

    def last_knn_ms(self) -> float:
        return float(lib().b200_map_last_knn_ms(self.h))

    def evicted(self) -> int:
        return int(lib().b200_map_evicted(self.h))

    def dropped(self):
        """(points dropped so far, by the last AddPoints) - non-finite or out-of-range points are skipped, not inserted."""
        last = C.c_int64(0)
        tot = lib().b200_map_dropped(self.h, C.byref(last))
        return int(tot), int(last.value)

    def NumValidGrids(self) -> int:
        return int(lib().b200_map_num_voxels(self.h))

    def NumPoints(self) -> int:
        return int(lib().b200_map_num_points(self.h))


class Esekf:
    """Device-resident esekf + ObsModel with the reference's call names (esekfom.hpp:1526,1836-1848)."""

    def __init__(self, ivox: IVox, max_iter=3, plane_thr=0.1, extrinsic_est_en=False, R=0.001, limit=0.001,
                 filter_size_map=0.5):
        p = IekfParams()
        p.max_iter, p.plane_thr, p.extrinsic_est_en, p.R, p.filter_size_map = max_iter, plane_thr, int(extrinsic_est_en), R, filter_size_map
        for i in range(23):
            p.limit[i] = limit if np.isscalar(limit) else limit[i]
        self.params = p
        self.ivox = ivox
        self.h = C.c_void_p()
        _check(lib().b200_iekf_create(C.byref(p), ivox.h, C.byref(self.h)))
        self.x = np.zeros(26)
        self.P = np.eye(23)
        self.stats = IekfStats()
        self._n = 0

    def close(self):
        if getattr(self, "h", None):
            try:
                lib().b200_iekf_destroy(self.h)
            except TypeError:  # interpreter shutdown: module globals are already torn down
                pass
            self.h = None

    __del__ = close

    def change_x(self, x):
        self.x = np.array(x, dtype=np.float64)

    def change_P(self, P):
        self.P = np.array(P, dtype=np.float64)

    def get_x(self):
        return self.x

    def get_P(self):
        return self.P

    def update_iterated_dyn_share_modified(self, scan_body):
        """One IEKF measurement update on the downsampled body-frame scan; returns the status code."""
        scan = _cloud(scan_body)
        self._n = scan.shape[0]
        rc = lib().b200_iekf_update(self.h, _p(scan), scan.shape[0], scan.strides[0], _p(self.x), _p(self.P), C.byref(self.stats))
        return _check(rc, soft=(0, 1))

    def update_device(self, d_scan_ptr, n):
        """Same update with the scan already on the device (float4 per point)."""
        self._n = n
        rc = lib().b200_iekf_update_device(self.h, C.c_void_p(d_scan_ptr), n, _p(self.x), _p(self.P), C.byref(self.stats))
        return _check(rc, soft=(0, 1))

    def set_profiling(self, on):
        _check(lib().b200_iekf_set_profiling(self.h, int(on)))

    def kernel_times_ms(self):
        ms = (C.c_float * 17)()
        k = lib().b200_iekf_kernel_times(self.h, ms, 17)
        return [ms[i] for i in range(k)]

    def launch_modes(self):
        """(graph captures, graph replays, plain launch sequences) so far."""
        a, b, c = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        _check(lib().b200_iekf_launch_modes(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def io_bytes(self, n):
        a, b = C.c_int64(0), C.c_int64(0)
        _check(lib().b200_iekf_io_bytes(self.h, n, C.byref(a), C.byref(b)))
        return a.value, b.value

    def last_HtH(self, p):
        HtH = np.zeros((12, 12))
        Hth = np.zeros(12)
        x_in = np.zeros(26)
        _check(lib().b200_iekf_last_HtH(self.h, p, _p(HtH), _p(Hth), _p(x_in)))
        return HtH, Hth, x_in

    def ObsModel(self, scan_body, x, converge=True):
        scan = _cloud(scan_body)
        self._n = scan.shape[0]
        x = np.ascontiguousarray(x, dtype=np.float64)
        HtH = np.zeros((12, 12))
        Hth = np.zeros(12)
        ne = C.c_int32(0)
        rc = lib().b200_iekf_obs_model(self.h, _p(scan), scan.shape[0], scan.strides[0], _p(x), int(converge), _p(HtH), _p(Hth), C.byref(ne))
        _check(rc, soft=(0, 1))
        return rc, HtH, Hth, ne.value

    def point_state(self, n=None):
        n = self._n if n is None else n
        plane = np.empty((n, 4), np.float32)
        res = np.empty(n, np.float32)
        sel = np.empty(n, np.uint8)
        nn = np.empty((n, 5), np.int32)
        cnt = np.empty(n, np.int32)
        _check(lib().b200_iekf_point_state(self.h, n, _p(plane), _p(res), _p(sel), _p(nn), _p(cnt)))
        return dict(plane=plane, residual=res, selected=sel, nn_idx=nn, nn_count=cnt)

    def predict(self, steps, Q12):
        """esekf::predict over the IMU intervals of a scan (steps [K,8] = dt, offs_t, acc_avr, angvel_avr) on the device; updates
        x / P in place and returns the IMUpose_ list [K,22] for the undistortion pass."""
        steps = np.ascontiguousarray(steps, dtype=np.float64).reshape(-1, 8)
        Q12 = np.ascontiguousarray(Q12, dtype=np.float64)
        poses = np.zeros((len(steps), 22))
        self.x = np.ascontiguousarray(self.x, dtype=np.float64)
        self.P = np.ascontiguousarray(self.P, dtype=np.float64)
        _check(lib().b200_iekf_predict(self.h, _p(steps), len(steps), _p(Q12), _p(self.x), _p(self.P), _p(poses)))
        return poses

    def world_scan(self, x=None, cols=3):
        """laserCloudWorld of PublishFrameWorld: the last scan in the world frame at state x ([n, cols] float32, xyz first)."""
        x = np.ascontiguousarray(self.x if x is None else x, dtype=np.float64)
        out = np.zeros((self._n, cols), np.float32)
        n = C.c_int64(0)
        _check(lib().b200_iekf_world_scan(self.h, _p(x), _p(out), out.strides[0], self._n, C.byref(n)))
        return out[:n.value]

    def MapIncremental(self, x=None, ekf_inited=True):
        x = np.ascontiguousarray(self.x if x is None else x, dtype=np.float64)
        na, nd = C.c_int32(0), C.c_int32(0)
        _check(lib().b200_iekf_map_incremental(self.h, _p(x), int(ekf_inited), C.byref(na), C.byref(nd)))
        return na.value, nd.value


class NormalDistributionsTransform:
    """pclomp::NormalDistributionsTransform's surface (ndt_omp.h:117-261) on the GPU engine."""

    def __init__(self, device=0):
        self._p = NdtParams(1.0, 0.1, 0.55, 0.1, 35, 7, 6, 0.01)  # ctor defaults, ndt_omp_impl.hpp:47-65
        self._device = device
        self.h = None
        self._target = None
        self._source = None
        self.result = NdtResult()
        self._final = np.eye(4, dtype=np.float32)
        self._dirty = True

    def _handle(self):
        if self.h is None or self._dirty:
            if self.h is not None:
                lib().b200_ndt_destroy(self.h)
            self.h = C.c_void_p()
            _check(lib().b200_ndt_create(C.byref(self._p), self._device, C.byref(self.h)))
            self._dirty = False
            if self._target is not None:
                _check(lib().b200_ndt_set_target(self.h, _p(self._target), self._target.shape[0], self._target.strides[0]))
            if self._source is not None:
                _check(lib().b200_ndt_set_source(self.h, _p(self._source), self._source.shape[0], self._source.strides[0]))
        return self.h

    def close(self):
        if getattr(self, "h", None):
            try:
                lib().b200_ndt_destroy(self.h)
            except TypeError:  # interpreter shutdown: module globals are already torn down
                pass
            self.h = None

    __del__ = close

    def setResolution(self, r):
        self._p.resolution = r
        self._dirty = True

    def setStepSize(self, s):
        self._p.step_size = s
        self._dirty = True

    def setOutlierRatio(self, o):
        self._p.outlier_ratio = o
        self._dirty = True

    def setTransformationEpsilon(self, e):
        self._p.trans_eps = e
        self._dirty = True

    def setMaximumIterations(self, n):
        self._p.max_iter = n
        self._dirty = True

    def setNeighborhoodSearchMethod(self, m):
        self._p.search = {"KDTREE": 0, "DIRECT1": 1, "DIRECT7": 7, "DIRECT26": 27}.get(m, m)
        self._dirty = True

    def setNumThreads(self, n):  # accepted for source compatibility; the device decides
        pass

    def setInputTarget(self, cloud):
        self._target = _cloud(cloud)
        if self.h is not None and not self._dirty:
            _check(lib().b200_ndt_set_target(self.h, _p(self._target), self._target.shape[0], self._target.strides[0]))

    def setInputTargetReplicated(self, comm, cloud, n, root=0):
        """setInputTarget on every rank of `comm` from the cloud held by `root` (others pass None); n on all ranks."""
        h = self._handle()
        if cloud is not None:
            c = _cloud(cloud)
            _check(lib().b200_ndt_set_target_bcast(comm.h, h, _p(c), n, c.strides[0], root))
        else:
            _check(lib().b200_ndt_set_target_bcast(comm.h, h, None, n, 16, root))

    def setInputSource(self, cloud):
        self._source = _cloud(cloud)
        if self.h is not None and not self._dirty:
            _check(lib().b200_ndt_set_source(self.h, _p(self._source), self._source.shape[0], self._source.strides[0]))

    def align(self, guess=None):
        g = np.eye(4, dtype=np.float32) if guess is None else np.asarray(guess, dtype=np.float32)
        gcm = np.ascontiguousarray(g.T)
        out = np.zeros((4, 4), np.float32)
        rc = lib().b200_ndt_align(self._handle(), _p(gcm), _p(out), C.byref(self.result))
        _check(rc, soft=(0, 2))
        self._final = out.T.copy()
        return rc

    def hasConverged(self):
        return bool(self.result.converged)

    def getFinalTransformation(self):
        return self._final

    def getFitnessScore(self, max_range=1.7976931348623157e308, T=None):
        """pcl::Registration::getFitnessScore: mean squared exact-NN distance of the aligned source to the target."""
        s, nr = C.c_double(0), C.c_int64(0)
        t = None if T is None else np.ascontiguousarray(np.asarray(T, dtype=np.float32).T)
        _check(lib().b200_ndt_fitness_score(self._handle(), None if t is None else _p(t), max_range, C.byref(s), C.byref(nr)))
        self.fitness_in_range = nr.value
        return s.value

    def getFinalNumIteration(self):
        return self.result.iters

    def getMaxEigen(self):
        """ndt_omp.h:209-223: the largest eigenvalue of the final Hessian / 100000 (localization-lost heuristic)."""
        H = np.array(self.result.hessian, dtype=np.float64)
        out = C.c_double(0)
        _check(lib().b200_ndt_max_eigen(_p(H), C.byref(out)))
        return out.value

    def getTransformationProbability(self):
        return self.result.trans_probability

    def numVoxels(self):
        return int(lib().b200_ndt_num_voxels(self._handle()))

    def leaves(self):
        h = self._handle()
        n = lib().b200_ndt_leaves(h, 0, None, None, None, None, None)
        ids = np.empty(n, np.int64)
        npts = np.empty(n, np.int32)
        mean = np.empty((n, 3))
        cov = np.empty((n, 3, 3))
        icov = np.empty((n, 3, 3))
        lib().b200_ndt_leaves(h, n, _p(ids), _p(npts), _p(mean), _p(cov), _p(icov))
        return dict(ids=ids, npts=npts, mean=mean, cov=cov, icov=icov)

    def computeDerivatives(self, p6):
        p6 = np.ascontiguousarray(p6, dtype=np.float64)
        s = C.c_double(0)
        g = np.zeros(6)
        H = np.zeros((6, 6))
        _check(lib().b200_ndt_derivatives(self._handle(), _p(p6), C.byref(s), _p(g), _p(H)))
        return s.value, g, H

    def computeHessian(self, p6):
        p6 = np.ascontiguousarray(p6, dtype=np.float64)
        H = np.zeros((6, 6))
        _check(lib().b200_ndt_hessian(self._handle(), _p(p6), _p(H)))
        return H

    def newtonDirection(self, H, rhs, force_svd=False):
        """JacobiSVD(H).solve(rhs) as the device computes it; returns (x, path) with path 0 = elimination shortcut, 1 = Jacobi SVD."""
        H = np.ascontiguousarray(H, dtype=np.float64)
        rhs = np.ascontiguousarray(rhs, dtype=np.float64)
        x = np.zeros(6)
        path = C.c_int32(0)
        _check(lib().b200_ndt_newton_direction(self._handle(), _p(H), _p(rhs), int(force_svd), _p(x), C.byref(path)))
        return x, path.value

    def calculateScore(self, poses_cm16):
        """calculateScore (ndt_omp_impl.hpp:836-880) for a batch of poses ([h,16] column-major 4x4)."""
        poses = np.ascontiguousarray(poses_cm16, dtype=np.float32).reshape(-1, 16)
        s = np.zeros(poses.shape[0])
        _check(lib().b200_ndt_score_batch(self._handle(), _p(poses), poses.shape[0], _p(s)))
        return s

    def alignBatch(self, guesses_cm16):
        """align() from h independent initial guesses in one batch; returns (finals [h,4,4] row-major, results)."""
        g = np.ascontiguousarray(guesses_cm16, dtype=np.float32).reshape(-1, 16)
        h = g.shape[0]
        out = np.zeros((h, 16), np.float32)
        res = (NdtResult * h)()
        _check(lib().b200_ndt_align_batch(self._handle(), _p(g), h, _p(out), res))
        return out.reshape(h, 4, 4).transpose(0, 2, 1).copy(), res

    def grid(self):
        mn = np.zeros(3, np.int32)
        dv = np.zeros(3, np.int32)
        _check(lib().b200_ndt_grid(self._handle(), _p(mn), _p(dv)))
        return mn, dv

    def nbhd_total(self, p6):
        p6 = np.ascontiguousarray(p6, dtype=np.float64)
        return int(lib().b200_ndt_nbhd_total(self._handle(), _p(p6)))

    def last_ms(self):
        """Device time (CUDA events on the handle's stream) of the last set_target / align / score call."""
        return float(lib().b200_ndt_last_ms(self._handle()))

    def last_launches(self):
        return int(lib().b200_ndt_last_launches(self._handle()))

    def last_score_kernel_ms(self):
        """Device time of the k_ndt_score_batch launch of the last calculateScore / relocalize call."""
        return float(lib().b200_ndt_last_score_kernel_ms(self._handle()))

    def score_pairs(self, poses_cm16):
        """(point, occupied voxel) pairs summed over the poses - roofline bookkeeping."""
        poses = np.ascontiguousarray(poses_cm16, dtype=np.float32).reshape(-1, 16)
        n = C.c_int64(0)
        _check(lib().b200_ndt_score_pairs(self._handle(), _p(poses), poses.shape[0], C.byref(n)))
        return n.value

    def stream_barrier(self, comm):
        """Device-side rendezvous of the ranks on this handle's stream (no-op without a communicator)."""
        _check(lib().b200_ndt_stream_barrier(comm.h if comm is not None else None, self._handle()))


class NdtPairBatch:
    """Registration of P independent (source, target, guess) pairs in one call - the loop-closure gate of
    mapOptmization.cpp:683-693 (a fresh NDT per candidate, align(guess), hasConverged() && getFitnessScore() <= threshold)
    for a whole batch of candidates.  Keyword arguments are the NDT setters: resolution, step_size, outlier_ratio,
    trans_eps, max_iter, search ("KDTREE" / "DIRECT1" / "DIRECT7" / "DIRECT26" or 0 / 1 / 7 / 27), min_pts, eig_ratio."""

    _DEFAULTS = dict(resolution=1.0, step_size=0.1, outlier_ratio=0.55, trans_eps=0.1, max_iter=35, search=7, min_pts=6, eig_ratio=0.01)

    def __init__(self, device=0, **setters):
        kw = dict(self._DEFAULTS)
        unknown = set(setters) - set(kw)
        if unknown:
            raise TypeError(f"unknown NDT parameter(s): {sorted(unknown)}")
        kw.update(setters)
        kw["search"] = {"KDTREE": 0, "DIRECT1": 1, "DIRECT7": 7, "DIRECT26": 27}.get(kw["search"], kw["search"])
        self._p = NdtParams(kw["resolution"], kw["step_size"], kw["outlier_ratio"], kw["trans_eps"], kw["max_iter"], kw["search"],
                            kw["min_pts"], kw["eig_ratio"])
        self.h = C.c_void_p()
        _check(lib().b200_ndt_pairs_create(C.byref(self._p), device, C.byref(self.h)))

    def close(self):
        if getattr(self, "h", None):
            try:
                lib().b200_ndt_pairs_destroy(self.h)
            except TypeError:  # interpreter shutdown: module globals are already torn down
                pass
            self.h = None

    __del__ = close

    @staticmethod
    def pack(clouds):
        """A list of [n_i, 3+] clouds -> (one contiguous float32 [sum n_i, 3] array, int64 offsets [P + 1])."""
        clouds = [np.asarray(c, dtype=np.float32) for c in clouds]
        clouds = [c.reshape(-1, 3) if c.ndim == 1 else c[:, :3] for c in clouds]
        off = np.zeros(len(clouds) + 1, np.int64)
        off[1:] = np.cumsum([len(c) for c in clouds])
        xyz = np.ascontiguousarray(np.concatenate(clouds, 0) if off[-1] else np.zeros((1, 3), np.float32), dtype=np.float32)
        return xyz, off

    def align(self, sources, targets, guesses=None, max_range=1.7976931348623157e308, comm=None):
        """Registers pair p = (sources[p], targets[p], guesses[p] (4x4 row-major; None = identity)).  Returns a dict of
        per-pair arrays: status, converged, iters, evals, hess_evals, final [P,4,4] (row-major), fitness, n_in_range, p_final
        [P,6], trans_probability, score, gpu_ms, and the raw ctypes records under "records"."""
        if len(sources) != len(targets):
            raise ValueError("sources and targets differ in length")
        P = len(sources)
        src, soff = self.pack(sources)
        tgt, toff = self.pack(targets)
        g = None
        if guesses is not None:
            g = np.ascontiguousarray(np.stack([np.asarray(m, dtype=np.float32).T.reshape(16) for m in guesses]), dtype=np.float32)
            if g.shape[0] != P:
                raise ValueError("one guess per pair")
        return self.align_packed(src, soff, tgt, toff, P, g, max_range, comm)

    def align_packed(self, src, soff, tgt, toff, P, guesses_cm16=None, max_range=1.7976931348623157e308, comm=None):
        """align() on clouds already in the offset layout of b200_ndt_pairs_align (guesses_cm16 = [P,16] column-major)."""
        res = (NdtPairResult * max(P, 1))()
        soff = np.ascontiguousarray(soff, dtype=np.int64)
        toff = np.ascontiguousarray(toff, dtype=np.int64)
        rc = lib().b200_ndt_pairs_align(comm.h if comm is not None else None, self.h, _p(src), _p(soff), _p(tgt), _p(toff), src.strides[0], P,
                                        None if guesses_cm16 is None else _p(guesses_cm16), max_range, res)
        _check(rc)
        return self.unpack(res, P)

    @staticmethod
    def unpack(res, P):
        out = dict(records=res)
        out["status"] = np.array([r.status for r in res[:P]], np.int32)
        out["converged"] = np.array([r.ndt.converged for r in res[:P]], np.int32)
        out["iters"] = np.array([r.ndt.iters for r in res[:P]], np.int32)
        out["evals"] = np.array([r.ndt.evals for r in res[:P]], np.int32)
        out["hess_evals"] = np.array([r.ndt.hess_evals for r in res[:P]], np.int32)
        out["final"] = np.array([np.array(r.final16, np.float32).reshape(4, 4).T for r in res[:P]], np.float32).reshape(P, 4, 4)
        out["fitness"] = np.array([r.fitness for r in res[:P]])
        out["n_in_range"] = np.array([r.n_in_range for r in res[:P]], np.int64)
        out["p_final"] = np.array([list(r.ndt.p_final) for r in res[:P]]).reshape(P, 6)
        out["trans_probability"] = np.array([r.ndt.trans_probability for r in res[:P]])
        out["score"] = np.array([r.ndt.score for r in res[:P]])
        out["gpu_ms"] = float(res[0].ndt.gpu_ms) if P else 0.0
        return out

    def leaves(self, p):
        """The valid leaves of pair p's target from the last align() (as NormalDistributionsTransform.leaves()), or None
        when pair p was not built in the last chunk of that call on this rank."""
        n = lib().b200_ndt_pairs_leaves(self.h, p, 0, None, None, None, None, None)
        if n < 0:
            return None
        ids = np.empty(n, np.int64)
        npts = np.empty(n, np.int32)
        mean = np.empty((n, 3))
        cov = np.empty((n, 3, 3))
        icov = np.empty((n, 3, 3))
        lib().b200_ndt_pairs_leaves(self.h, p, n, _p(ids), _p(npts), _p(mean), _p(cov), _p(icov))
        return dict(ids=ids, npts=npts, mean=mean, cov=cov, icov=icov)


class Communicator:
    """NCCL communicator over the ranks of a torch.distributed-style job (one process per GPU)."""

    def __init__(self, nranks, rank, unique_id: bytes, device=0):
        self.h = C.c_void_p()
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        _check(lib().b200_comm_init_rank(nranks, rank, buf, device, C.byref(self.h)))
        self.nranks, self.rank = nranks, rank

    @staticmethod
    def unique_id() -> bytes:
        buf = (C.c_uint8 * 128)()
        _check(lib().b200_comm_unique_id(buf))
        return bytes(buf)

    def close(self):
        if getattr(self, "h", None):
            try:
                lib().b200_comm_destroy(self.h)
            except TypeError:  # interpreter shutdown: module globals are already torn down
                pass
            self.h = None

    __del__ = close


def shard_range(h_total: int, nranks: int, rank: int):
    """Contiguous slice [begin, end) of h_total hypotheses owned by `rank` (sizes differ by at most one)."""
    base, rem = divmod(h_total, nranks)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


# ---- host-side statement of the map builder's merge protocol (b200_mapbuild_merge, csrc/voxel.cu): used by the CPU tests that run
# the N > 1 path over gloo; the product path is the CUDA + NCCL implementation, this is only its contract in numpy
def voxel_key(cells) -> "np.ndarray":
    """pack_key(cz, cy, cx) of csrc/common.cuh for an [n, 3] array of (cx, cy, cz) voxel cells (21-bit biased fields)."""
    c = np.asarray(cells, dtype=np.int64) + (1 << 20)
    return (c[:, 2].astype(np.uint64) << np.uint64(42)) | (c[:, 1].astype(np.uint64) << np.uint64(21)) | c[:, 0].astype(np.uint64)


def voxel_owner(keys, nranks: int) -> "np.ndarray":
    """owner_of(key, nranks) of csrc/voxel.cu: the rank that holds a voxel after the merge."""
    k = np.asarray(keys, dtype=np.uint64) ^ np.uint64(0x9E3779B97F4A7C15)
    with np.errstate(over="ignore"):
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xff51afd7ed558ccd)
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xc4ceb9fe1a85ec53)
        k ^= k >> np.uint64(33)
    return (((k & np.uint64(0xFFFFFFFF)) >> np.uint64(8)) % np.uint64(nranks)).astype(np.int64)


def mapbuild_merge_protocol_host(keys, counts, sums, nranks: int, rank: int, exchange):
    """One rank's side of the merge: records (key, count, sums[4]) are routed to their owner and records of the same voxel are
    added.  `exchange(list_of_per_destination_arrays)` returns the list of arrays received from every rank (an all-to-all).
    Returns the (keys, counts, sums) this rank owns afterwards, sorted by key."""
    owner = voxel_owner(keys, nranks)
    rec = np.concatenate([np.asarray(keys, np.uint64).view(np.float64)[:, None], np.asarray(counts, np.float64)[:, None], np.asarray(sums, np.float64)], 1)
    got = np.concatenate(exchange([rec[owner == r] for r in range(nranks)]), 0)
    k = got[:, 0].copy().view(np.uint64)
    uniq, inv = np.unique(k, return_inverse=True)
    cnt = np.zeros(len(uniq))
    sm = np.zeros((len(uniq), got.shape[1] - 2))
    np.add.at(cnt, inv, got[:, 1])
    np.add.at(sm, inv, got[:, 2:])
    return uniq, cnt.astype(np.int64), sm


def score_key(s: float) -> int:
    """Order-preserving map fp64 -> uint64 used by the allreduce-argmin (NaN -> 0, below every real score)."""
    import struct
    if s != s:
        return 0
    u = struct.unpack("<Q", struct.pack("<d", s))[0]
    return (~u) & 0xFFFFFFFFFFFFFFFF if (u >> 63) else (u | (1 << 63))


def score_from_key(k: int) -> float:
    import struct
    u = (k & 0x7FFFFFFFFFFFFFFF) if (k >> 63) else ((~k) & 0xFFFFFFFFFFFFFFFF)
    return struct.unpack("<d", struct.pack("<Q", u))[0]


def argmin_protocol_host(scores, h_begin, all_gather):
    """Host mirror of b200_reloc_argmin's collective protocol (used by the CPU gloo test): every rank contributes its local
    winner as an (order-preserving score key, global index) pair; all_gather(tensor[2]) returns the pairs of all ranks
    ([R, 2] int64, keys shifted into int64 order by xor 2^63 because gloo has no uint64); the global winner is the pair
    with the highest key, ties to the lowest index."""
    import torch
    keys = [score_key(float(s)) for s in scores]
    lk, li = 0, (1 << 62)
    for i, k in enumerate(keys):
        if k > lk:
            lk, li = k, h_begin + i
    pairs = all_gather(torch.tensor([lk - (1 << 63), li], dtype=torch.int64))
    best_k, best_i = 0, (1 << 62)
    for kr, ir in pairs.tolist():
        kr += (1 << 63)
        if kr > best_k or (kr == best_k and kr != 0 and ir < best_i):
            best_k, best_i = kr, ir
    if best_k == 0 or best_i == (1 << 62):
        return -1, 0.0
    return best_i, score_from_key(best_k)


def relocalize(ndt: "NormalDistributionsTransform", poses_cm16, comm: Communicator | None = None, h_begin=0, h_stride=1):
    """Global relocalization: scores this rank's hypothesis slice (poses_cm16 = the slice; local hypothesis i is global
    hypothesis h_begin + i * h_stride) and returns (global best index, its score, device ms) - identical on every rank.
    Contiguous slices: h_begin = shard_range(...)[0]; interleaved slices: poses[rank::nranks], h_begin = rank, h_stride = nranks."""
    poses = np.ascontiguousarray(poses_cm16, dtype=np.float32).reshape(-1, 16)
    best, score, ms = C.c_int64(-1), C.c_double(0), C.c_float(0)
    rc = lib().b200_reloc_argmin_strided(comm.h if comm is not None else None, ndt._handle(), _p(poses) if len(poses) else None,
                                         poses.shape[0], h_begin, h_stride, C.byref(best), C.byref(score), C.byref(ms))
    _check(rc)
    return best.value, score.value, ms.value


class VoxelGrid:
    """pcl::VoxelGrid's surface (setLeafSize / setInputCloud / filter) on the GPU (laser_mapping.cc:323-328)."""

    def __init__(self, device=0):
        self.h = C.c_void_p()
        _check(lib().b200_downsampler_create(device, C.byref(self.h)))
        self.leaf, self.min_points = 0.5, 0
        self._cloud = None

    def close(self):
        if getattr(self, "h", None):
            try:
                lib().b200_downsampler_destroy(self.h)
            except TypeError:  # interpreter shutdown: module globals are already torn down
                pass
            self.h = None

    __del__ = close

    def setLeafSize(self, lx, ly=None, lz=None):
        self.leaf = float(lx)

    def setMinimumPointsNumberPerVoxel(self, n):
        self.min_points = int(n)

    def setInputCloud(self, cloud):
        a = np.asarray(cloud)
        self._cloud = np.ascontiguousarray(a, dtype=np.float32)

    def filter(self):
        """Returns (centroids [m,4] x y z intensity, counts [m])."""
        a = self._cloud
        n = a.shape[0]
        out = np.empty((max(n, 1), 4), np.float32)
        cnt = np.empty(max(n, 1), np.int32)
        m = C.c_int64(0)
        _check(lib().b200_voxel_downsample(self.h, _p(a), n, a.strides[0], self.leaf, self.min_points, _p(out), _p(cnt), n, C.byref(m)))
        return out[:m.value].copy(), cnt[:m.value].copy()

    def undistort(self, points, time_index, intensity_index, poses22, x_end26, want_host=True):
        """ImuProcess::UndistortPcl (backward half) on the raw scan; the result stays staged on the device.
        Returns (xyzi [n,4] in time order, order [n]) when want_host."""
        a = np.ascontiguousarray(points, dtype=np.float32)
        poses = np.ascontiguousarray(poses22, dtype=np.float64).reshape(-1, 22)
        x = np.ascontiguousarray(x_end26, dtype=np.float64)
        n = a.shape[0]
        out = np.zeros((n, 4), np.float32) if want_host else None
        order = np.zeros(n, np.int32) if want_host else None
        _check(lib().b200_scan_undistort(self.h, _p(a), n, a.strides[0], time_index, intensity_index, _p(poses), poses.shape[0], _p(x),
                                         _p(out) if want_host else None, _p(order) if want_host else None))
        return out, order

    def filter_staged(self):
        """VoxelGrid on the staged (undistorted) scan; returns the number of voxels (result on the device)."""
        m = C.c_int64(0)
        _check(lib().b200_voxel_downsample_staged(self.h, self.leaf, self.min_points, C.byref(m)))
        return m.value

    def device_points(self):
        n = C.c_int64(0)
        p = lib().b200_downsampler_device_points(self.h, C.byref(n))
        return p, n.value

    def last_ms(self):
        return float(lib().b200_downsampler_last_ms(self.h))


class FullMapBuilder:
    """construct_full_map <poses.txt> <frames_dir> <out.pcd> <leaf>: keyframes + poses -> voxel-grid merged map."""

    def __init__(self, leaf=0.1, capacity_voxels=8_000_000, device=0):
        self.h = C.c_void_p()
        _check(lib().b200_mapbuild_create(leaf, capacity_voxels, device, C.byref(self.h)))

    def close(self):
        if getattr(self, "h", None):
            try:
                lib().b200_mapbuild_destroy(self.h)
            except TypeError:  # interpreter shutdown: module globals are already torn down
                pass
            self.h = None

    __del__ = close

    def add_keyframe(self, xyzi, pose7):
        a = np.ascontiguousarray(xyzi, dtype=np.float32)
        p = np.ascontiguousarray(pose7, dtype=np.float64)
        _check(lib().b200_mapbuild_add_keyframe(self.h, _p(a), a.shape[0], a.strides[0], _p(p)))

    def add_keyframe_device(self, d_ptr, n, pose7):
        p = np.ascontiguousarray(pose7, dtype=np.float64)
        _check(lib().b200_mapbuild_add_keyframe_device(self.h, C.c_void_p(d_ptr), n, _p(p)))

    def add_keyframes_device(self, d_ptrs, ns, poses7):
        """A batch of device-resident keyframes (pointers, point counts, count x 7 poses) in one call."""
        ptrs = np.ascontiguousarray(d_ptrs, dtype=np.uint64)
        ns = np.ascontiguousarray(ns, dtype=np.int64)
        p = np.ascontiguousarray(poses7, dtype=np.float64).reshape(-1, 7)
        assert len(ptrs) == len(ns) == len(p)
        _check(lib().b200_mapbuild_add_keyframes_device(self.h, _p(ptrs), _p(ns), _p(p), len(ptrs)))

    def num_voxels(self):
        n = lib().b200_mapbuild_num_voxels(self.h)
        if n < 0:
            raise B200Error(lib().b200_last_error().decode())
        return int(n)

    def merge(self, comm):
        _check(lib().b200_mapbuild_merge(comm.h if comm is not None else None, self.h))

    def exchange_ms(self):
        return float(lib().b200_mapbuild_last_exchange_ms(self.h))

    def extract(self):
        m = lib().b200_mapbuild_extract(self.h, None, None, 0)
        if m < 0:
            raise B200Error(lib().b200_last_error().decode())
        out = np.empty((max(m, 1), 4), np.float32)
        cnt = np.empty(max(m, 1), np.int32)
        lib().b200_mapbuild_extract(self.h, _p(out), _p(cnt), m)
        return out[:m].copy(), cnt[:m].copy()


class ScanToMap:
    """jueying_slam mapOptimization's scan2MapOptimization on the GPU (mapOptmization.cpp:1255-1590).
    Transforms are transformTobeMapped: (roll, pitch, yaw, x, y, z) float32."""

    def __init__(self, max_map_points=2_000_000, device=0):
        self.h = C.c_void_p()
        _check(lib().b200_loam_create(max_map_points, device, C.byref(self.h)))
        self.stats = LoamStats()

    def close(self):
        if getattr(self, "h", None):
            try:
                lib().b200_loam_destroy(self.h)
            except TypeError:  # interpreter shutdown: module globals are already torn down
                pass
            self.h = None

    __del__ = close

    def setInputCloud(self, corner_map, surf_map):
        c, s = _cloud(corner_map), _cloud(surf_map)
        _check(lib().b200_loam_set_map(self.h, _p(c), c.shape[0], c.strides[0], _p(s), s.shape[0], s.strides[0]))

    def scan2MapOptimization(self, corner, surf, t6, iter_num=30):
        c, s = _cloud(corner), _cloud(surf)
        t = np.array(t6, dtype=np.float32)
        rc = lib().b200_loam_optimize(self.h, _p(c), c.shape[0], c.strides[0], _p(s), s.shape[0], s.strides[0], _p(t), iter_num, C.byref(self.stats))
        _check(rc, soft=(0, 2))
        return t, rc

    def features(self, corner, surf, t6):
        c, s = _cloud(corner), _cloud(surf)
        t = np.ascontiguousarray(t6, dtype=np.float32)
        n = len(c) + len(s)
        flags = np.zeros(n, np.uint8)
        coeff = np.zeros((n, 4), np.float32)
        nsel = C.c_int32(0)
        _check(lib().b200_loam_features(self.h, _p(c), c.shape[0], c.strides[0], _p(s), s.shape[0], s.strides[0], _p(t), _p(flags), _p(coeff), C.byref(nsel)))
        return nsel.value, flags, coeff


class GeneralizedIterativeClosestPoint:
    """pclomp::GeneralizedIterativeClosestPoint's surface (gicp_omp.h:60-283 + the pcl::Registration calls
    jueying_slam/src/localization.cpp:277,323-328 makes) on the GPU engine."""

    def __init__(self, device=0):
        self._p = GicpParams(20, 0.001, 2e-3, 5e-4, 5.0, 200, 20)  # ctor defaults, gicp_omp.h:115-127
        self._device = device
        self.h = None
        self._target = None
        self._source = None
        self.result = GicpResult()
        self._final = np.eye(4, dtype=np.float32)
        self._dirty = True

    def _handle(self):
        if self.h is None or self._dirty:
            if self.h is not None:
                lib().b200_gicp_destroy(self.h)
            self.h = C.c_void_p()
            _check(lib().b200_gicp_create(C.byref(self._p), self._device, C.byref(self.h)))
            self._dirty = False
            if self._target is not None:
                _check(lib().b200_gicp_set_target(self.h, _p(self._target), self._target.shape[0], self._target.strides[0]))
            if self._source is not None:
                _check(lib().b200_gicp_set_source(self.h, _p(self._source), self._source.shape[0], self._source.strides[0]))
        return self.h

    def close(self):
        if getattr(self, "h", None):
            try:
                lib().b200_gicp_destroy(self.h)
            except TypeError:  # interpreter shutdown
                pass
            self.h = None

    __del__ = close

    def _set(self, name, v):
        setattr(self._p, name, v)
        self._dirty = True

    def setCorrespondenceRandomness(self, k):
        self._set("k_correspondences", int(k))

    def setRotationEpsilon(self, e):
        self._set("rotation_epsilon", float(e))

    def setTransformationEpsilon(self, e):
        self._set("transformation_epsilon", float(e))

    def setMaxCorrespondenceDistance(self, d):
        self._set("corr_dist_threshold", float(d))

    def setMaximumIterations(self, n):
        self._set("max_iterations", int(n))

    def setMaximumOptimizerIterations(self, n):
        self._set("max_inner_iterations", int(n))

    def setInputTarget(self, cloud):
        self._target = _cloud(cloud)
        if self.h is not None and not self._dirty:
            _check(lib().b200_gicp_set_target(self.h, _p(self._target), self._target.shape[0], self._target.strides[0]))

    def setInputSource(self, cloud):
        self._source = _cloud(cloud)
        if self.h is not None and not self._dirty:
            _check(lib().b200_gicp_set_source(self.h, _p(self._source), self._source.shape[0], self._source.strides[0]))

    def align(self, guess=None):
        g = np.eye(4, dtype=np.float32) if guess is None else np.asarray(guess, dtype=np.float32)
        gcm = np.ascontiguousarray(g.T)
        out = np.zeros((4, 4), np.float32)
        rc = lib().b200_gicp_align(self._handle(), _p(gcm), _p(out), C.byref(self.result))
        _check(rc, soft=(0, 2))
        self._final = out.T.copy()
        return rc

    def hasConverged(self):
        return bool(self.result.converged)

    def getFinalTransformation(self):
        return self._final

    def getFitnessScore(self, max_range=1.7976931348623157e308, T=None):
        s, nr = C.c_double(0), C.c_int64(0)
        t = None if T is None else np.ascontiguousarray(np.asarray(T, dtype=np.float32).T)
        _check(lib().b200_gicp_fitness_score(self._handle(), None if t is None else _p(t), max_range, C.byref(s), C.byref(nr)))
        self.fitness_in_range = nr.value
        return s.value

    # parity probes
    def covariances(self, which, with_neighbours=False):
        cloud = self._target if which == "target" else self._source
        n = cloud.shape[0]
        cov = np.zeros((n, 3, 3))
        knn = np.zeros((n, self._p.k_correspondences), np.int32) if with_neighbours else None
        _check(lib().b200_gicp_covariances(self._handle(), 1 if which == "target" else 0, _p(cov), None if knn is None else _p(knn)))
        return (cov, knn) if with_neighbours else cov

    def correspondences(self, trans=None, guess=None):
        t = np.ascontiguousarray((np.eye(4) if trans is None else np.asarray(trans)).T, dtype=np.float32)
        g = np.ascontiguousarray((np.eye(4) if guess is None else np.asarray(guess)).T, dtype=np.float32)
        n = self._source.shape[0]
        idx = np.zeros(n, np.int32)
        maha = np.zeros((n, 3, 3), np.float32)
        d2 = np.zeros(n, np.float32)
        m = C.c_int64(0)
        _check(lib().b200_gicp_correspondences(self._handle(), _p(t), _p(g), _p(idx), _p(maha), _p(d2), C.byref(m)))
        return m.value, idx, maha, d2

    def cost(self, x6):
        x = np.ascontiguousarray(x6, dtype=np.float64)
        f0, f1, m = C.c_double(), C.c_double(), C.c_int64()
        g = np.zeros(6)
        _check(lib().b200_gicp_cost(self._handle(), _p(x), C.byref(f0), C.byref(f1), _p(g), C.byref(m)))
        return f0.value, f1.value, g, m.value

    def index_info(self, which):
        leaf, cells, occ = C.c_float(), C.c_int64(), C.c_int64()
        _check(lib().b200_gicp_index_info(self._handle(), 1 if which == "target" else 0, C.byref(leaf), C.byref(cells), C.byref(occ)))
        return dict(leaf=leaf.value, cells=cells.value, occupied=occ.value)
