// TEST INFRASTRUCTURE ONLY — CPU oracle for the LOAM local map built from the keyframe store (b200_loam_set_map_from_keyframes).
// PARITY UNPINNED (see oracle.h): the reference is extractSurroundingKeyFrames of LIO-SAM's published mapOptmization.cpp, from
// which jueying_slam derives; it is not in the tree.  Restated here:
//   extractNearby: kdtreeSurroundingKeyPoses->radiusSearch(cloudKeyPoses3D->back(), surroundingKeyframeSearchRadius) over the
//     keyframe positions (hits in ascending (distance, index) order); downSizeFilterSurroundingKeyPoses (VoxelGrid with leaf
//     surroundingKeyframeDensity) of the hits in that order; each centroid's intensity becomes the index of its nearest
//     keyframe (nearestKSearch(pt, 1) over all of cloudKeyPoses3D, ties to the lower index); then the keyframes newest
//     first while timeLaserInfoCur - time < 10.0, stopping at the first that fails, appended even when already listed;
//   extractCloud: an entry farther than surroundingKeyframeSearchRadius from cloudKeyPoses3D->back() (pointDistance = sqrt of
//     the squared distance) is skipped; the others append transformPointCloud(corner / surf cloud, pose) to
//     laserCloud{Corner,Surf}FromMap; downSizeFilterCorner (mappingCornerLeafSize) and downSizeFilterSurf
//     (mappingSurfLeafSize) give laserCloud{Corner,Surf}FromMapDS.  The laserCloudMapContainer cache holds the same values.
// Third-party arithmetic restated from published behaviour (versions unpinned), as in loop_oracle.cpp:
//   pcl::KdTreeFLANN: squared distance L2_Simple<float> (float differences, squares summed x, y, z left to right), radius
//     test strictly below (float)(radius * radius) in double; equal distances in ascending index order;
//   pcl::getTransformation: the explicit ZYX matrix in float, sin / cos as correctly rounded floats (loam_oracle.cpp);
//   pcl::VoxelGrid: orc_voxel_grid (voxelgrid_oracle.cpp), min points 0.
#include "oracle.h"

#include <algorithm>
#include <cmath>
#include <utility>
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

float sqdist(const float* a, const float* b) {  // FLANN L2_Simple<float>: float differences, squares summed x, y, z
    float d = 0.f;
    for (int k = 0; k < 3; ++k) {
        const float diff = a[k] - b[k];
        d += diff * diff;
    }
    return d;
}
void append_moved(const float* xyzi, int64_t lo, int64_t hi, const float* p6, std::vector<float>& all) {
    float T[12];
    pose_matrix(p6, T);
    for (int64_t i = lo; i < hi; ++i) {
        const float* p = xyzi + 4 * i;
        all.push_back(T[0] * p[0] + T[1] * p[1] + T[2] * p[2] + T[3]);
        all.push_back(T[4] * p[0] + T[5] * p[1] + T[6] * p[2] + T[7]);
        all.push_back(T[8] * p[0] + T[9] * p[1] + T[10] * p[2] + T[11]);
        all.push_back(p[3]);
    }
}
}  // namespace

extern "C" {
void orc_loam_surrounding(const float* xyzi, const int64_t* offsets, const int64_t* n_corner, const float* poses6, const double* times, int64_t cur,
                          double time_cur, const float* prm4, int64_t* keys, int64_t* n_keys, int64_t* n_list, float* corner_out, int64_t* n_c,
                          float* surf_out, int64_t* n_s, int64_t max_out);
}

extern "C" {
/* extractSurroundingKeyFrames with keyframe cur the newest (keyframes 0 .. cur exist): prm4 = search_radius, density, corner_leaf,
 * surf_leaf.  Keyframe k's cloud is xyzi records offsets[k] .. offsets[k+1]-1, its first n_corner[k] the corner cloud.  keys
 * (room for 2 (cur + 1)) / *n_keys: the list after the distance gate; *n_list its length before; the downsampled maps (4 floats
 * per point, at most max_out each) and their sizes. */
void orc_loam_surrounding(const float* xyzi, const int64_t* offsets, const int64_t* n_corner, const float* poses6, const double* times, int64_t cur,
                          double time_cur, const float* prm4, int64_t* keys, int64_t* n_keys, int64_t* n_list, float* corner_out, int64_t* n_c,
                          float* surf_out, int64_t* n_s, int64_t max_out) {
    const float radius = prm4[0], density = prm4[1];
    const float r2 = (float)((double)radius * (double)radius);
    const float* q = poses6 + 6 * cur;
    std::vector<std::pair<float, int64_t>> hits;
    for (int64_t j = 0; j <= cur; ++j) {
        const float d = sqdist(q, poses6 + 6 * j);
        if (d < r2) hits.push_back({d, j});
    }
    std::sort(hits.begin(), hits.end());
    std::vector<float> pos;
    for (const auto& h : hits)
        for (int k = 0; k < 4; ++k) pos.push_back(k < 3 ? poses6[6 * h.second + k] : 0.f);
    const int64_t nh = (int64_t)hits.size();
    std::vector<float> cent(4 * std::max<int64_t>(nh, 1));
    std::vector<int32_t> ccnt(std::max<int64_t>(nh, 1));
    const int64_t ncent = nh ? orc_voxel_grid(pos.data(), nh, 16, density, 0, cent.data(), ccnt.data(), nh) : 0;
    std::vector<std::pair<int64_t, std::vector<float>>> list;  // (keyframe, point of the entry)
    for (int64_t c = 0; c < ncent; ++c) {
        const float* pc = &cent[4 * c];
        int64_t best = 0;
        float bd = sqdist(pc, poses6);
        for (int64_t j = 1; j <= cur; ++j) {
            const float d = sqdist(pc, poses6 + 6 * j);
            if (d < bd) { bd = d; best = j; }
        }
        list.push_back({best, {pc[0], pc[1], pc[2]}});
    }
    for (int64_t j = cur; j >= 0; --j) {
        if (!(time_cur - times[j] < 10.0)) break;
        list.push_back({j, {poses6[6 * j], poses6[6 * j + 1], poses6[6 * j + 2]}});
    }
    *n_list = (int64_t)list.size();
    std::vector<float> corner, surf;
    int64_t nk = 0;
    for (const auto& e : list) {
        if (std::sqrt(sqdist(e.second.data(), q)) > radius) continue;
        const int64_t k = e.first;
        keys[nk++] = k;
        append_moved(xyzi, offsets[k], offsets[k] + n_corner[k], poses6 + 6 * k, corner);
        append_moved(xyzi, offsets[k] + n_corner[k], offsets[k + 1], poses6 + 6 * k, surf);
    }
    *n_keys = nk;
    std::vector<int32_t> cnt(std::max<int64_t>(max_out, 1));
    const int64_t mc = (int64_t)corner.size() / 4, ms = (int64_t)surf.size() / 4;
    *n_c = mc ? orc_voxel_grid(corner.data(), mc, 16, prm4[2], 0, corner_out, cnt.data(), max_out) : 0;
    *n_s = ms ? orc_voxel_grid(surf.data(), ms, 16, prm4[3], 0, surf_out, cnt.data(), max_out) : 0;
}
}
