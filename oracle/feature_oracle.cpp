// TEST INFRASTRUCTURE ONLY — CPU oracle for the LOAM front end on the device (b200_features_extract): imageProjection's
// projection and extraction, featureExtraction and mapOptimization's downsampleCurrentScan.
// PARITY UNPINNED (see oracle.h): the reference is LIO-SAM's published imageProjection.cpp / featureExtraction.cpp /
// mapOptmization.cpp, from which jueying_slam derives; none of them is in the tree.  Restated here (this is the contract):
//   parameters  N_SCAN, Horizon_SCAN, downsampleRate, lidarMinRange, lidarMaxRange, edgeThreshold, surfThreshold,
//               odometrySurfLeafSize, mappingCornerLeafSize, mappingSurfLeafSize; sensor velodyne/ouster (column from the
//               azimuth) or livox (column = arrival order within the line).
//   input       records of `stride` bytes, x y z the first three floats, intensity a float at a byte offset (absent: 0), the
//               ring an unsigned 1- or 2-byte integer at a byte offset; points in input order.
//   1 projectPointCloud (no deskew: deskewFlag == -1, the stored point is the input point unchanged), per point in order:
//     a point with a non-finite coordinate is dropped; range = sqrtf((x*x + y*y) + z*z) (fp32, no FMA), dropped unless
//     minRange <= range <= maxRange; row = ring, dropped when row >= N_SCAN or row % downsampleRate != 0; column:
//     velodyne/ouster  horizonAngle = (float)((double)(atan2f(x, y) * 180.0f) / M_PI), ang_res_x = (float)(360.0 / (float)H),
//                      col = (int)(-round(((double)horizonAngle - 90.0) / ang_res_x) + H / 2), col -= H when col >= H
//                      (atan2f = fp64 atan2 narrowed to float, the project's libm rule; round = half away from zero);
//     livox            col = a per-row counter (reset every scan) incremented by every point that passed range and row;
//     dropped when col < 0 or col >= H; the first point of a pixel wins.
//   2 cloudExtraction: row-major walk, startRingIndex[i] = count - 1 + 5 at the start of row i, occupied pixels appended in
//     column order with pointColInd and pointRange, endRingIndex[i] = count - 1 - 5 at its end.
//   3 calculateSmoothness for 5 <= i < size - 5: diffRange = r[i-5] + .. + r[i-1] - r[i] * 10 + r[i+1] + .. + r[i+5] (fp32, left
//     to right), curvature = diffRange^2, picked = label = 0, sort entry (curvature, i).
//   4 markOccludedPoints for 5 <= i < size - 6: |col[i+1] - col[i]| < 10 and (double)(r[i] - r[i+1]) > 0.3 marks i-5 .. i, else
//     (double)(r[i+1] - r[i]) > 0.3 marks i+1 .. i+6; fabsf(r[i-1] - r[i]) > 0.02 * (double)r[i] and the same for i+1 marks i.
//   5 extractFeatures: per ring, six regions sp = (S(6-j) + E j) / 6, ep = (S(5-j) + E(j+1)) / 6 - 1 (C++ int division), skipped
//     when sp >= ep; entries [sp, ep) sorted by curvature; corner pass k = ep .. sp (at most 20 picks, the 21st candidate ends
//     it), surf pass k = sp .. ep (curvature < surfThreshold, label -1), both marking neighbours (picked[ind] = 1, then up to 5
//     each side, stopping at a column jump > 10); the ring's surf list = points sp .. ep with label <= 0, VoxelGrid
//     (odometrySurfLeafSize) per ring, appended in ascending leaf order.
//   6 downsampleCurrentScan: VoxelGrid(mappingCornerLeafSize) of cornerCloud, VoxelGrid(mappingSurfLeafSize) of surfaceCloud.
// Quirks, defined here as DESIGN.md §2 lists them:
//   1 std::sort is not stable: the order is (curvature, index) ascending, so among equal curvatures the corner pass takes the
//     higher index first.
//   2 stale state: every index outside [5, size - 5) has curvature 0, picked 0, label 0 and sort entry (0, i) at the start of
//     each scan (the reference reads uninitialised memory and earlier scans' sort entries at index 4).
//   3 position ep of each region is outside the sort; both passes visit it.
//   4 endRingIndex itself lies in no region (never a feature), nor do the points of skipped regions.
//   5 a neighbour walk that would read below index 0 stops there (the reference reads pointColInd[-1]).
//   6 rings never interact in step 5 (S_{i+1} - E_i = 10): marks of ring i stay within [S_i - 5, E_i + 4].
//   7 the azimuth: see DESIGN.md §2; the column follows from the float bits of horizonAngle.
// VoxelGrid is orc_voxel_grid (voxelgrid_oracle.cpp), min points 0.
#include "oracle.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <utility>
#include <vector>

namespace {

float rd_f(const uint8_t* p) {
    float v;
    memcpy(&v, p, 4);
    return v;
}

// neighbour marking of extractFeatures, shared by the corner and surf passes
void mark_neighbours(int64_t ind, int64_t m, const std::vector<int32_t>& col, std::vector<uint8_t>& picked) {
    picked[ind] = 1;
    for (int l = 1; l <= 5; ++l) {
        if (ind + l >= m) break;
        if (std::abs(col[ind + l] - col[ind + l - 1]) > 10) break;
        picked[ind + l] = 1;
    }
    for (int l = -1; l >= -5; --l) {
        if (ind + l < 0) break;
        if (std::abs(col[ind + l] - col[ind + l + 1]) > 10) break;
        picked[ind + l] = 1;
    }
}

}  // namespace

extern "C" {
int64_t orc_features(const uint8_t* pts, int64_t n, int64_t stride, int64_t int_off, int64_t ring_off, int32_t ring_bytes, const int32_t* iprm,
                     const float* fprm, float* cloud, int32_t* col_out, float* range_out, int32_t* start_out, int32_t* end_out, float* curv_out,
                     int8_t* label_out, uint8_t* picked_out, float* corner, float* surface, float* corner_ds, float* surf_ds, int64_t* counts);
}

extern "C" {
/* Steps 1-6 for one scan.  iprm = N_SCAN, Horizon_SCAN, downsampleRate, sensor (0 velodyne/ouster, 1 livox); fprm = minRange,
 * maxRange, edgeThreshold, surfThreshold, odometrySurfLeafSize, mappingCornerLeafSize, mappingSurfLeafSize.  int_off < 0: no
 * intensity.  Outputs (the caller gives room for n points each; start / end N_SCAN each): the extracted cloud (4 floats per
 * point), pointColInd, pointRange, start / endRingIndex, curvature, label, picked, cornerCloud (pick order), surfaceCloud, and
 * the two DS clouds.  counts = dropped non-finite, range, row, column, duplicate pixel; extracted, corner, surface, cornerDS,
 * surfDS.  Returns the extracted size. */
int64_t orc_features(const uint8_t* pts, int64_t n, int64_t stride, int64_t int_off, int64_t ring_off, int32_t ring_bytes, const int32_t* iprm,
                     const float* fprm, float* cloud, int32_t* col_out, float* range_out, int32_t* start_out, int32_t* end_out, float* curv_out,
                     int8_t* label_out, uint8_t* picked_out, float* corner, float* surface, float* corner_ds, float* surf_ds, int64_t* counts) {
    const int N = iprm[0], H = iprm[1], rate = iprm[2], livox = iprm[3];
    const float min_r = fprm[0], max_r = fprm[1], edge = fprm[2], surf_th = fprm[3];
    for (int k = 0; k < 10; ++k) counts[k] = 0;
    // 1 projection
    std::vector<int64_t> owner((size_t)N * H, -1);
    std::vector<float> rmat((size_t)N * H, 0.f);
    std::vector<int32_t> livox_cnt(N, 0);
    const float ang_res_x = (float)(360.0 / (float)H);
    for (int64_t i = 0; i < n; ++i) {
        const uint8_t* p = pts + i * stride;
        const float x = rd_f(p), y = rd_f(p + 4), z = rd_f(p + 8);
        if (!std::isfinite(x) || !std::isfinite(y) || !std::isfinite(z)) { ++counts[0]; continue; }
        const float range = std::sqrt((x * x + y * y) + z * z);
        if (range < min_r || range > max_r) { ++counts[1]; continue; }
        const int row = ring_bytes == 1 ? (int)p[ring_off] : (int)(p[ring_off] | (p[ring_off + 1] << 8));
        if (row >= N || row % rate != 0) { ++counts[2]; continue; }
        int c;
        if (livox) {
            c = livox_cnt[row]++;
        } else {
            const float a = (float)std::atan2((double)x, (double)y);
            const float horizon = (float)((double)(a * 180.0f) / M_PI);
            c = (int)(-std::round(((double)horizon - 90.0) / (double)ang_res_x) + H / 2);
            if (c >= H) c -= H;
        }
        if (c < 0 || c >= H) { ++counts[3]; continue; }
        const size_t pix = (size_t)row * H + c;
        if (owner[pix] >= 0) { ++counts[4]; continue; }
        owner[pix] = i;
        rmat[pix] = range;
    }
    // 2 extraction
    std::vector<int32_t> col;
    std::vector<float> r;
    int64_t m = 0;
    for (int i = 0; i < N; ++i) {
        start_out[i] = (int32_t)(m - 1 + 5);
        for (int j = 0; j < H; ++j) {
            const size_t pix = (size_t)i * H + j;
            if (owner[pix] < 0) continue;
            const uint8_t* p = pts + owner[pix] * stride;
            cloud[4 * m] = rd_f(p); cloud[4 * m + 1] = rd_f(p + 4); cloud[4 * m + 2] = rd_f(p + 8);
            cloud[4 * m + 3] = int_off >= 0 ? rd_f(p + int_off) : 0.f;
            col.push_back(j);
            r.push_back(rmat[pix]);
            ++m;
        }
        end_out[i] = (int32_t)(m - 1 - 5);
    }
    counts[5] = m;
    for (int64_t i = 0; i < m; ++i) { col_out[i] = col[i]; range_out[i] = r[i]; }
    // 3 smoothness (quirk 2: zero state outside [5, m - 5))
    std::vector<float> curv(m, 0.f);
    std::vector<uint8_t> picked(m, 0);
    std::vector<int8_t> label(m, 0);
    std::vector<std::pair<float, int64_t>> ent(m);
    for (int64_t i = 0; i < m; ++i) ent[i] = {0.f, i};
    for (int64_t i = 5; i < m - 5; ++i) {
        const float d = r[i - 5] + r[i - 4] + r[i - 3] + r[i - 2] + r[i - 1] - r[i] * 10 + r[i + 1] + r[i + 2] + r[i + 3] + r[i + 4] + r[i + 5];
        curv[i] = d * d;
        ent[i] = {curv[i], i};
    }
    // 4 occlusion and parallel beams
    for (int64_t i = 5; i < m - 6; ++i) {
        const float d1 = r[i], d2 = r[i + 1];
        if (std::abs(col[i + 1] - col[i]) < 10) {
            if ((double)(d1 - d2) > 0.3) {
                for (int k = 0; k <= 5; ++k) picked[i - k] = 1;
            } else if ((double)(d2 - d1) > 0.3) {
                for (int k = 1; k <= 6; ++k) picked[i + k] = 1;
            }
        }
        const float df1 = std::fabs(r[i - 1] - r[i]), df2 = std::fabs(r[i + 1] - r[i]);
        if (df1 > 0.02 * (double)r[i] && df2 > 0.02 * (double)r[i]) picked[i] = 1;
    }
    // 5 features
    std::vector<float> corner_v, surface_v, ring_surf;
    std::vector<int32_t> vcnt(std::max<int64_t>(m, 1));
    std::vector<float> vout(4 * std::max<int64_t>(m, 1));
    for (int i = 0; i < N; ++i) {
        ring_surf.clear();
        const int64_t S = start_out[i], E = end_out[i];
        for (int j = 0; j < 6; ++j) {
            const int64_t sp = (S * (6 - j) + E * j) / 6, ep = (S * (5 - j) + E * (j + 1)) / 6 - 1;
            if (sp >= ep) continue;
            std::sort(ent.begin() + sp, ent.begin() + ep);  // pairs: (curvature, index) ascending (quirk 1)
            int largest = 0;
            for (int64_t k = ep; k >= sp; --k) {
                const int64_t ind = ent[k].second;
                if (picked[ind] == 0 && curv[ind] > edge) {
                    if (++largest > 20) break;
                    label[ind] = 1;
                    for (int q = 0; q < 4; ++q) corner_v.push_back(cloud[4 * ind + q]);
                    mark_neighbours(ind, m, col, picked);
                }
            }
            for (int64_t k = sp; k <= ep; ++k) {
                const int64_t ind = ent[k].second;
                if (picked[ind] == 0 && curv[ind] < surf_th) {
                    label[ind] = -1;
                    mark_neighbours(ind, m, col, picked);
                }
            }
            for (int64_t k = sp; k <= ep; ++k)
                if (label[k] <= 0)
                    for (int q = 0; q < 4; ++q) ring_surf.push_back(cloud[4 * k + q]);
        }
        const int64_t ns = (int64_t)ring_surf.size() / 4;
        const int64_t nd = ns ? orc_voxel_grid(ring_surf.data(), ns, 16, fprm[4], 0, vout.data(), vcnt.data(), m) : 0;
        surface_v.insert(surface_v.end(), vout.begin(), vout.begin() + 4 * nd);
    }
    for (int64_t i = 0; i < m; ++i) { curv_out[i] = curv[i]; label_out[i] = label[i]; picked_out[i] = picked[i]; }
    const int64_t nc = (int64_t)corner_v.size() / 4, ns = (int64_t)surface_v.size() / 4;
    std::copy(corner_v.begin(), corner_v.end(), corner);
    std::copy(surface_v.begin(), surface_v.end(), surface);
    counts[6] = nc;
    counts[7] = ns;
    // 6 downsampleCurrentScan
    counts[8] = nc ? orc_voxel_grid(corner, nc, 16, fprm[5], 0, corner_ds, vcnt.data(), m) : 0;
    counts[9] = ns ? orc_voxel_grid(surface, ns, 16, fprm[6], 0, surf_ds, vcnt.data(), m) : 0;
    return m;
}
}
