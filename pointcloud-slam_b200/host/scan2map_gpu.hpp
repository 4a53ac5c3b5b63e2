// b200reg host adaptor — jueying_slam's scan-to-map step and the scan pre-processing chain on top of the C ABI.
//
// ScanToMap mirrors the members mapOptimization uses around scan2MapOptimization (jueying_slam/src/mapOptmization.cpp:1560-1590):
// the two feature maps (kdtree{Corner,Surf}FromMap->setInputCloud) and transformTobeMapped[6] = roll, pitch, yaw, x, y, z.
// FeatureExtraction runs imageProjection / featureExtraction / downsampleCurrentScan (LIO-SAM) on raw scans, clouds left on the device.
// ScanPreprocessor chains ImuProcess::UndistortPcl's backward half (jueying_lio/include/imu_processing.hpp:247-284) and
// pcl::VoxelGrid::filter (jueying_lio/src/laser_mapping.cc:323-328) on the device.
#pragma once
#include "ivox_gpu.hpp"

namespace b200host {

template <typename CloudT>
class ScanToMap {
   public:
    explicit ScanToMap(int64_t max_map_points = 2000000, int device = 0) { check(b200_loam_create(max_map_points, device, &h_), "b200_loam_create"); }
    ~ScanToMap() { b200_loam_destroy(h_); }
    ScanToMap(const ScanToMap&) = delete;
    ScanToMap& operator=(const ScanToMap&) = delete;

    /// kdtreeCornerFromMap->setInputCloud(laserCloudCornerFromMapDS); kdtreeSurfFromMap->setInputCloud(laserCloudSurfFromMapDS)
    void setInputCloud(const CloudT& corner_map, const CloudT& surf_map) {
        using P = typename std::remove_reference<decltype(corner_map.points[0])>::type;
        check(b200_loam_set_map(h_, corner_map.points.empty() ? nullptr : &corner_map.points[0].x, (int64_t)corner_map.points.size(), sizeof(P),
                                surf_map.points.empty() ? nullptr : &surf_map.points[0].x, (int64_t)surf_map.points.size(), sizeof(P)),
              "b200_loam_set_map");
    }
    /// extractSurroundingKeyFrames from a device keyframe store (b200host::KeyframeStore, ndt_gpu.hpp; cur = -1: its last keyframe)
    /// followed by setInputCloud, the two maps never leaving the device; false when the store is empty (the maps stay)
    template <class Store>
    bool extractSurroundingKeyFrames(Store& store, int64_t cur, double timeLaserInfoCur, const b200_surround_params& params) {
        const int32_t rc = b200_loam_set_map_from_keyframes(h_, store.handle(), cur, timeLaserInfoCur, &params, &info_);
        check(rc, "b200_loam_set_map_from_keyframes");
        return rc == B200_OK;
    }
    const b200_surround_info& surroundInfo() const { return info_; }
    /// the iterCount loop of scan2MapOptimization; returns LMOptimization's convergence flag, isDegenerate in degenerate()
    bool scan2MapOptimization(const CloudT& corner_last_ds, const CloudT& surf_last_ds, float transformTobeMapped[6], int iter_num = 30) {
        using P = typename std::remove_reference<decltype(corner_last_ds.points[0])>::type;
        const int32_t rc = b200_loam_optimize(h_, corner_last_ds.points.empty() ? nullptr : &corner_last_ds.points[0].x, (int64_t)corner_last_ds.points.size(),
                                              sizeof(P), surf_last_ds.points.empty() ? nullptr : &surf_last_ds.points[0].x,
                                              (int64_t)surf_last_ds.points.size(), sizeof(P), transformTobeMapped, iter_num, &stats_);
        check(rc, "b200_loam_optimize");
        return rc == B200_OK;
    }
    /// the same on laserCloud{Corner,Surf}LastDS as FeatureExtraction left them on the device (deviceCloud)
    bool scan2MapOptimization(const void* d_corner_last_ds, int64_t n_corner, const void* d_surf_last_ds, int64_t n_surf, float transformTobeMapped[6],
                              int iter_num = 30) {
        const int32_t rc = b200_loam_optimize_device(h_, d_corner_last_ds, n_corner, d_surf_last_ds, n_surf, transformTobeMapped, iter_num, &stats_);
        check(rc, "b200_loam_optimize_device");
        return rc == B200_OK;
    }
    bool degenerate() const { return stats_.degenerate != 0; }
    const b200_loam_stats& stats() const { return stats_; }

   private:
    b200_loam* h_ = nullptr;
    b200_loam_stats stats_{};
    b200_surround_info info_{};
};

/// imageProjection (projection and cloud extraction, no deskew), featureExtraction and downsampleCurrentScan on the device for
/// raw scans of PointT (x, y, z and intensity floats, an unsigned 1- or 2-byte `ring`, as velodyne / ouster / livox point types
/// carry them); the four clouds stay on the device for ScanToMap::scan2MapOptimization and KeyframeStore::add
template <typename PointT>
class FeatureExtraction {
   public:
    explicit FeatureExtraction(const b200_feature_params& params, int device = 0) { check(b200_features_create(&params, device, &h_), "b200_features_create"); }
    ~FeatureExtraction() { b200_features_destroy(h_); }
    FeatureExtraction(const FeatureExtraction&) = delete;
    FeatureExtraction& operator=(const FeatureExtraction&) = delete;

    /// one scan (laserCloudIn in input order); false when no point survives the projection (empty clouds)
    template <typename Alloc>
    bool extract(const std::vector<PointT, Alloc>& scan) {
        static_assert(sizeof(PointT{}.ring) == 1 || sizeof(PointT{}.ring) == 2, "ring must be a 1- or 2-byte unsigned integer");
        const PointT p{};
        const int64_t int_off = (const char*)&p.intensity - (const char*)&p, ring_off = (const char*)&p.ring - (const char*)&p;
        const int32_t rc = b200_features_extract(h_, scan.empty() ? nullptr : scan.data(), (int64_t)scan.size(), sizeof(PointT), int_off, ring_off,
                                                 (int32_t)sizeof(p.ring), &info_);
        check(rc, "b200_features_extract");
        return rc == B200_OK;
    }
    const b200_feature_info& info() const { return info_; }
    /// B200_FEATURES_CORNER / SURFACE / CORNER_DS / SURF_DS as float4 (x, y, z, intensity) on the device, valid until the next extract
    const void* deviceCloud(int which, int64_t* n) const { return b200_features_device_cloud(h_, which, n); }
    /// a copy on the host (x y z intensity per point)
    std::vector<float> cloud(int which) const {
        int64_t n = 0;
        b200_features_device_cloud(h_, which, &n);
        std::vector<float> out(4 * (size_t)n);
        check(b200_features_cloud(h_, which, out.data(), n, &n), "b200_features_cloud");
        return out;
    }

   private:
    b200_features* h_ = nullptr;
    b200_feature_info info_{};
};

/// raw scan -> (undistort) -> voxel downsample, result left on the device for Esekf::update on device points
class ScanPreprocessor {
   public:
    explicit ScanPreprocessor(int device = 0) { check(b200_downsampler_create(device, &h_), "b200_downsampler_create"); }
    ~ScanPreprocessor() { b200_downsampler_destroy(h_); }
    ScanPreprocessor(const ScanPreprocessor&) = delete;
    ScanPreprocessor& operator=(const ScanPreprocessor&) = delete;

    /// IMUpose = std::vector<common::Pose6D> of the forward propagation (22 doubles each); x_end26 = kf_state.get_x() after the last predict
    template <typename PointVector>
    void undistort(const PointVector& scan, int time_index, int intensity_index, const double* imu_pose22, int n_poses, const double* x_end26) {
        using P = typename PointVector::value_type;
        check(b200_scan_undistort(h_, reinterpret_cast<const float*>(scan.data()), (int64_t)scan.size(), sizeof(P), time_index, intensity_index, imu_pose22,
                                  n_poses, x_end26, nullptr, nullptr),
              "b200_scan_undistort");
    }
    /// voxel_scan_.filter(*scan_down_body_) on the staged (undistorted) scan; returns the number of downsampled points
    int64_t filterStaged(float leaf) {
        int64_t n = 0;
        check(b200_voxel_downsample_staged(h_, leaf, 0, &n), "b200_voxel_downsample_staged");
        return n;
    }
    /// device pointer (float4 per point) and size of the downsampled scan: pass to b200_iekf_update_device
    const void* devicePoints(int64_t* n) const { return b200_downsampler_device_points(h_, n); }

   private:
    b200_downsampler* h_ = nullptr;
};

}  // namespace b200host
