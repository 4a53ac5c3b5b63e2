// TEST INFRASTRUCTURE ONLY — CPU oracle for the front half of the loop closure.
// PARITY UNPINNED (see oracle.h): the reference's loop closure is LIO-SAM's published mapOptmization.cpp, from which
// jueying_slam derives; it is not in the tree.  Restated here:
//   detectLoopClosureDistance: kdtreeHistoryKeyPoses->radiusSearch(newest keyframe, historyKeyframeSearchRadius) over the
//     keyframe positions, then the first hit (ascending distance) with |time - time_newest| > historyKeyframeSearchTimeDiff;
//   loopFindNearKeyframes(key, searchNum): keyframes key-searchNum .. key+searchNum clipped to the store, each moved by
//     transformPointCloud(cloud, &cloudKeyPoses6D[k]) and appended in index order, then downSizeFilterICP (VoxelGrid).
// Third-party arithmetic restated from published behaviour (versions unpinned):
//   pcl::KdTreeFLANN::radiusSearch: exact (FLANN, eps 0, unlimited checks), squared distance L2_Simple<float> (float
//     differences, squares summed x, y, z left to right) strictly below (float)(radius * radius) in double, results sorted
//     by distance; equal distances are taken in ascending index order (the project's FLANN tie contract);
//   pcl::getTransformation: the explicit ZYX matrix in float, sin / cos as correctly rounded floats (loam_oracle.cpp);
//   pcl::VoxelGrid: orc_voxel_grid (voxelgrid_oracle.cpp), min points 0.
#include "oracle.h"

#include <algorithm>
#include <cmath>
#include <vector>

namespace {

inline float fsin(float a) { return (float)std::sin((double)a); }
inline float fcos(float a) { return (float)std::cos((double)a); }

void pose_matrix(const float* p6, float* T) {  // p6 = x y z roll pitch yaw (PointTypePose)
    const float roll = p6[3], pitch = p6[4], yaw = p6[5];
    const float A = fcos(yaw), B = fsin(yaw), C = fcos(pitch), D = fsin(pitch), E = fcos(roll), F = fsin(roll), DE = D * E, DF = D * F;
    T[0] = A * C; T[1] = A * DF - B * E; T[2] = B * F + A * DE; T[3] = p6[0];
    T[4] = B * C; T[5] = A * E + B * DF; T[6] = B * DE - A * F; T[7] = p6[1];
    T[8] = -D;    T[9] = C * F;          T[10] = C * E;         T[11] = p6[2];
}

}  // namespace

extern "C" {
void orc_loop_detect(const float* poses6, const double* times, int64_t K, const int64_t* cur, int64_t Q, float radius, double time_gap,
                     int64_t* pre, float* sqdist);
int64_t orc_loop_submap(const float* xyzi, const int64_t* offsets, const float* poses6, int64_t K, int64_t key, int32_t num, float leaf,
                        float* raw_xyzi, int64_t* n_raw, float* out_xyzi, int32_t* out_count, int64_t max);

/* detectLoopClosureDistance with cur[q] as the newest keyframe (only keyframes j < cur[q] exist then): pre[q] (-1 = none),
 * sqdist[q] (0 = none) */
void orc_loop_detect(const float* poses6, const double* times, int64_t K, const int64_t* cur, int64_t Q, float radius, double time_gap,
                     int64_t* pre, float* sqdist) {
    (void)K;
    const float r2 = (float)((double)radius * (double)radius);
    for (int64_t q = 0; q < Q; ++q) {
        const int64_t c = cur[q];
        const float* a = poses6 + 6 * c;
        int64_t best = -1;
        float bd = 0.f;
        for (int64_t j = 0; j < c; ++j) {
            const float* b = poses6 + 6 * j;
            float d = 0.f;
            for (int k = 0; k < 3; ++k) {
                const float diff = a[k] - b[k];
                d += diff * diff;
            }
            if (!(d < r2) || !(std::fabs(times[j] - times[c]) > time_gap)) continue;
            if (best < 0 || d < bd) { best = j; bd = d; }
        }
        pre[q] = best;
        sqdist[q] = best < 0 ? 0.f : bd;
    }
}

/* loopFindNearKeyframes(key, num): keyframe k = xyzi records offsets[k] .. offsets[k+1]-1 (4 floats each) with pose
 * poses6[k].  raw_xyzi (may be NULL, room for every raw point) receives the concatenation, *n_raw its size; out_xyzi /
 * out_count the VoxelGrid(leaf) result (at most max written); returns the number of downsampled points. */
int64_t orc_loop_submap(const float* xyzi, const int64_t* offsets, const float* poses6, int64_t K, int64_t key, int32_t num, float leaf,
                        float* raw_xyzi, int64_t* n_raw, float* out_xyzi, int32_t* out_count, int64_t max) {
    std::vector<float> all;
    for (int64_t k = key - num; k <= key + num; ++k) {
        if (k < 0 || k >= K) continue;
        float T[12];
        pose_matrix(poses6 + 6 * k, T);
        for (int64_t i = offsets[k]; i < offsets[k + 1]; ++i) {
            const float* p = xyzi + 4 * i;
            all.push_back(T[0] * p[0] + T[1] * p[1] + T[2] * p[2] + T[3]);
            all.push_back(T[4] * p[0] + T[5] * p[1] + T[6] * p[2] + T[7]);
            all.push_back(T[8] * p[0] + T[9] * p[1] + T[10] * p[2] + T[11]);
            all.push_back(p[3]);
        }
    }
    const int64_t n = (int64_t)all.size() / 4;
    if (n_raw) *n_raw = n;
    if (raw_xyzi && n) std::copy(all.begin(), all.end(), raw_xyzi);
    if (!n) return 0;
    return orc_voxel_grid(all.data(), n, 16, leaf, 0, out_xyzi, out_count, max);
}
}
