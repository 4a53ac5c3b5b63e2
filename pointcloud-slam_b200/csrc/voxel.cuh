// b200reg — what the VoxelGrid downsample (voxel.cu) shares with the segmented downsample of the loop-closure submaps
// (loop.cu): the grid of a cloud and the per-leaf centroid kernel.
#pragma once
#include "common.cuh"

namespace b200 {
namespace vox {

struct Grid {
    long long min_b[3], div_b[3];
    float inv_leaf;
};

// applyFilter's grid (voxel_grid_large.cpp:67-103) from the min / max of the finite points (ordered ints, as the min / max
// kernels leave them): cells = leaves of the grid, 0 when there is no finite point; B200_ERR_RANGE past 9e18 leaves
int32_t grid_from_minmax(const int* mm6, float leaf, Grid& g, unsigned long long& cells);

// one thread per leaf: fp32 sums in input order, divided by the count (pcl::CentroidPoint); compacts on min_points
__global__ void k_centroids(const float4* __restrict__ pts, const int32_t* __restrict__ sorted_idx, const unsigned long long* __restrict__ uniq,
                            const int32_t* __restrict__ run_off, const int32_t* __restrict__ run_cnt, const int32_t* __restrict__ nruns,
                            unsigned long long sentinel, int min_points, float4* __restrict__ out, int32_t* __restrict__ out_cnt,
                            uint8_t* __restrict__ keep);

}  // namespace vox
}  // namespace b200
