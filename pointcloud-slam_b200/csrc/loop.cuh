// b200reg — the keyframe store's side of the loop closure (loop.cu), as the pair registration (ndt.cu) drives it.
#pragma once
#include "common.cuh"

#include <vector>

namespace b200 {
namespace ndt {
// Min / max of the finite points of segments: segment y = off[y] .. off[y+1]-1 of pts, into mm[6 y .. 6 y + 6) (ordered ints:
// min x y z, max x y z).  Defined in ndt.cu (the NDT target build); the submaps' VoxelGrid uses them too.
__global__ void k_ndt_minmax_init(int* mm, int np);
__global__ void k_ndt_minmax(const float4* __restrict__ pts, const int64_t* __restrict__ off, int* __restrict__ mm);
}  // namespace ndt

namespace loop {

struct Seg {  // loopFindNearKeyframes(key, num)
    int64_t key;
    int32_t num;
};
struct Part {  // points begin .. begin+count-1 of keyframe kf's cloud
    int64_t kf, begin, count;
};
struct GatherEntry {  // gather(): count points from pts[src ..) to dst[which][dst ..)
    int64_t src, count, dst;
    int64_t which;
};
struct Submaps {
    const float4* pts = nullptr;       // device: the downsampled points of every segment, segment after segment
    std::vector<int64_t> first, count; // per segment: its points are pts[first .. first + count)
    std::vector<int32_t> status;       // per segment: B200_OK, or the code b200_voxel_downsample returns for this cloud
    int64_t done = 0;                  // segments assembled: a prefix of whole groups
};

// scratch of the segmented VoxelGrid (seg_downsample), kept by its owner between calls
struct SegWork {
    PinnedBuf<uint8_t> h_tab;
    DevBuf<uint8_t> d_tab;
    DevBuf<int64_t> d_io;
    PinnedBuf<int64_t> h_io;
    DevBuf<float4> d_cent;
    DevBuf<int32_t> d_mm;
    PinnedBuf<int32_t> h_mm;
    DevBuf<unsigned long long> k_in, k_out, k_uniq;
    DevBuf<int32_t> v_in, v_out, run_cnt, run_off, d_cnt, d_small;
    DevBuf<uint8_t> keep, cub_tmp;
};

int32_t check_params(const b200_loop_params* prm);
// keys[0 .. n) in [0, count); with allow_none, -1 too
int32_t check_keys(const b200_keyframes* h, const int64_t* keys, int64_t n, bool allow_none);
int32_t device_of(const b200_keyframes* h);
// points of loopFindNearKeyframes(key, num) before the downsample
int64_t raw_size(const b200_keyframes* h, int64_t key, int32_t num);
// detectLoopClosureDistance for Q queries on stream s (one read-back)
int32_t detect(b200_keyframes* h, cudaStream_t s, const int64_t* cur, int64_t Q, const b200_loop_params& prm, int64_t* pre, float* sqdist);
// Assembles and VoxelGrid-downsamples segs[0 .. nseg) on stream s (two read-backs: min / max, run ranges).  Segments come in
// groups of `group`; the call ends after the last whole group whose leaves still fit the 64-bit sort key (at least one group).
// Out-of-range raw sizes are the caller's: the raw points of all segments must stay below 2^31.
int32_t submaps(b200_keyframes* h, cudaStream_t s, const Seg* segs, int64_t nseg, int64_t group, float leaf, Submaps& out);
// The same for general segments: segment j is parts[part_off[j] .. part_off[j+1]) appended in order, downsampled with leaf[j].
int32_t assemble(b200_keyframes* h, cudaStream_t s, const Part* parts, const int64_t* part_off, const float* leaf, int64_t nseg, int64_t group,
                 Submaps& out);
// The VoxelGrid half of assemble for device-resident segments: segment j = pts[off[j] .. off[j+1]) (off[0] = 0; d_off the same
// offsets on the device, outside w.d_tab's bytes from grid_at on, where the grids go), downsampled with leaf[j]; non-finite
// points are skipped.  Two read-backs (min / max, run ranges); out.pts = w.d_cent, valid until w is used again.
int32_t seg_downsample(SegWork& w, cudaStream_t s, const float4* pts, const int64_t* d_off, const int64_t* off, size_t grid_at, const float* leaf,
                       int64_t nseg, int64_t group, Submaps& out);
// loopFindNearKeyframes(key, num) as parts
void near_parts(const b200_keyframes* h, int64_t key, int32_t num, std::vector<Part>& parts);
// e[0 .. n) from pts into dst0 / dst1 as (x, y, z, 0) records, one launch on stream s
int32_t gather(b200_keyframes* h, cudaStream_t s, const float4* pts, const GatherEntry* e, int64_t n, float4* dst0, float4* dst1);
cudaStream_t stream_of(const b200_keyframes* h);

// extractSurroundingKeyFrames from the store (arguments checked by check_surround; cur = -1: the last keyframe): the keyframe
// list after extractCloud's distance gate, and the corner map (segment 0) and surf map (segment 1) downsampled with their
// leaves in out.sm.  One read-back of its own (the list; a list past 4096 entries takes one more copy) plus the two of
// assemble.  B200_NO_EFFECTIVE_POINTS on an empty store; a keyframe without a corner / surf split is B200_ERR_ARG; a
// key-pose or map grid out of range is B200_ERR_RANGE.
struct Surround {
    std::vector<int64_t> keys;  // the list after the gate, in extraction order
    int64_t n_list = 0;         // its length before the gate
    int64_t raw[2] = {0, 0};    // laserCloud{Corner,Surf}FromMap sizes
    Submaps sm;
};
int32_t check_surround(const b200_keyframes* h, int64_t cur, double time_cur, const b200_surround_params* prm);
int32_t surrounding(b200_keyframes* h, int64_t cur, double time_cur, const b200_surround_params& prm, Surround& out);

}  // namespace loop
}  // namespace b200
