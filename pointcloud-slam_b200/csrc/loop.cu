// b200reg — loop closure from a device keyframe store: the front half of performLoopClosure (LIO-SAM mapOptmization.cpp,
// from which jueying_slam derives; the registration half is mapOptmization.cpp:683-693, b200_ndt_pairs in ndt.cu).
//
// store        every keyframe cloud as float4 (x, y, z, intensity) records end to end in one device pool with int64 offsets;
//              one record per keyframe {pcl::getTransformation of its pose (float 3x4), time} in a device array.  A pose
//              update (correctPoses) rewrites the records only.
// detection    detectLoopClosureDistance: one warp per query scans keyframes 0 .. q-1 and keeps the lexicographic minimum of
//              (squared distance bits, index) over the keyframes inside the radius and outside the time gap - exact, and
//              ties go to the lower index.  10^5 keyframes x 10^3 queries is 10^8 distance tests: no index is needed.
// submaps      loopFindNearKeyframes for a batch of submaps: one gather kernel moves every keyframe of every submap into
//              the world frame (transformPointCloud, fp32, no FMA) straight from the pool through a (keyframe, offset)
//              table, then ONE segmented VoxelGrid: per-segment min / max (k_ndt_minmax) -> per-segment grid on the host as
//              b200_voxel_downsample derives it -> key = segment base + leaf index (the bases lay the segments' cell ranges
//              end to end, one sentinel sorts last) -> one stable radix sort -> run-length encoding + scan -> k_centroids.
//              A segment's output is therefore what b200_voxel_downsample returns for its cloud alone, bit for bit.
//              A segment is a list of (keyframe, sub-range) parts with its own leaf, so the LOAM local map (corner map and
//              surf map, two leaves) is one more caller of the same assembly.
// local map    extractSurroundingKeyFrames (mapOptmization.cpp, LIO-SAM): radius hits of the newest keyframe marked and
//              sorted by (d2 bits, index), the key-pose VoxelGrid on the device (grid from a device min / max, the vox::
//              key and centroid arithmetic), one warp per centroid for its nearest keyframe (k_loop_detect's distance and
//              ties), the 10 s recent walk and the distance gate; the ordered list is read back once and becomes the
//              assembly table of two segments.
#include "common.cuh"
#include "loop.cuh"
#include "voxel.cuh"

#include <cub/cub.cuh>

#include <algorithm>
#include <cmath>
#include <vector>

namespace b200 {
namespace loop {

struct KfRec {      // one keyframe on the device
    float T[12];    // pcl::getTransformation(x, y, z, roll, pitch, yaw), row-major 3x4: T[3], T[7], T[11] = x, y, z
    double time;
};
struct AsmEntry {   // one keyframe of one submap
    int64_t kf, src, n, dst;
};
struct SegGrid {
    long long min_b[3], div_b[3];
    unsigned long long base;  // keys of this segment: base + leaf index
    long long live;           // 0: no finite point or grid out of range; the points take the sentinel
    float inv_leaf;           // 1.0f / leaf of this segment
    int pad;
};

// pcl::getTransformation (PCL common/eigen.hpp) in float, sin / cos as the correctly rounded floats (fp64, narrowed)
static void pose_matrix(const float* p6, float* T) {
    const auto fs = [](float a) { return (float)std::sin((double)a); };
    const auto fc = [](float a) { return (float)std::cos((double)a); };
    const float roll = p6[3], pitch = p6[4], yaw = p6[5];
    const float A = fc(yaw), B = fs(yaw), C = fc(pitch), D = fs(pitch), E = fc(roll), F = fs(roll), DE = D * E, DF = D * F;
    T[0] = A * C; T[1] = A * DF - B * E; T[2] = B * F + A * DE; T[3] = p6[0];
    T[4] = B * C; T[5] = A * E + B * DF; T[6] = B * DE - A * F; T[7] = p6[1];
    T[8] = -D;    T[9] = C * F;          T[10] = C * E;         T[11] = p6[2];
}

// FLANN's L2_Simple<float> (float differences, squares summed x, y, z left to right), strict radius test (RadiusResultSet)
__global__ void k_loop_detect(const KfRec* __restrict__ rec, const int64_t* __restrict__ cur, int Q, float r2, double gap, int64_t* __restrict__ pre,
                              float* __restrict__ sqdist) {
    const int w = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (w >= Q) return;
    const int64_t q = cur[w];
    const float qx = rec[q].T[3], qy = rec[q].T[7], qz = rec[q].T[11];
    const double tq = rec[q].time;
    unsigned long long best = ~0ull;
    for (int64_t j = lane; j < q; j += 32) {
        const KfRec& r = rec[j];
        const float dx = __fsub_rn(qx, r.T[3]), dy = __fsub_rn(qy, r.T[7]), dz = __fsub_rn(qz, r.T[11]);
        const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
        if (d2 < r2 && fabs(r.time - tq) > gap) best = min(best, ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned long long)j);
    }
    for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
    if (lane == 0) {
        pre[w] = best == ~0ull ? -1 : (int64_t)(best & 0xffffffffull);
        sqdist[w] = best == ~0ull ? 0.f : __uint_as_float((unsigned)(best >> 32));
    }
}

// transformPointCloud (mapOptmization.cpp): T(r,0) x + T(r,1) y + T(r,2) z + T(r,3), left to right, no FMA; intensity copied.
// One block per (submap, keyframe) entry.
__global__ void __launch_bounds__(256) k_loop_assemble(const float4* __restrict__ pool, const KfRec* __restrict__ rec, const AsmEntry* __restrict__ ent,
                                                       float4* __restrict__ out) {
    const AsmEntry e = ent[blockIdx.x];
    float T[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) T[k] = rec[e.kf].T[k];
    for (int64_t i = threadIdx.x; i < e.n; i += blockDim.x) {
        const float4 p = __ldg(pool + e.src + i);
        float4 o;
        o.x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[0], p.x), __fmul_rn(T[1], p.y)), __fmul_rn(T[2], p.z)), T[3]);
        o.y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[4], p.x), __fmul_rn(T[5], p.y)), __fmul_rn(T[6], p.z)), T[7]);
        o.z = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[8], p.x), __fmul_rn(T[9], p.y)), __fmul_rn(T[10], p.z)), T[11]);
        o.w = p.w;
        out[e.dst + i] = o;
    }
}

// leaf index of every point of segment blockIdx.y (vox::k_keys' arithmetic) plus the segment's base; non-finite points and
// segments that are not live get the sentinel
__global__ void k_loop_keys(const float4* __restrict__ pts, const int64_t* __restrict__ off, const SegGrid* __restrict__ sg,
                            unsigned long long sentinel, unsigned long long* __restrict__ keys, int32_t* __restrict__ vals) {
    const int64_t b = off[blockIdx.y], n = off[blockIdx.y + 1] - b;
    const SegGrid g = sg[blockIdx.y];
    const float inv_leaf = g.inv_leaf;
#pragma unroll 1
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 p = __ldg(pts + b + i);
        unsigned long long key = sentinel;
        if (g.live && isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) {
            const long long i0 = (long long)(floorf(p.x * inv_leaf) - (float)g.min_b[0]);
            const long long i1 = (long long)(floorf(p.y * inv_leaf) - (float)g.min_b[1]);
            const long long i2 = (long long)(floorf(p.z * inv_leaf) - (float)g.min_b[2]);
            key = g.base + (unsigned long long)(i0 + i1 * g.div_b[0] + i2 * g.div_b[0] * g.div_b[1]);
        }
        keys[b + i] = key;
        vals[b + i] = (int32_t)(b + i);
    }
}

__device__ __forceinline__ int64_t lower_bound_u64(const unsigned long long* a, int64_t n, unsigned long long v) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}
// the runs of segment s are those whose key lies in [base, base + cells): first and count of them
__global__ void k_loop_seg_runs(const unsigned long long* __restrict__ uniq, const int32_t* __restrict__ nruns, const SegGrid* __restrict__ sg,
                                const unsigned long long* __restrict__ cells, int nseg, int64_t* __restrict__ fc) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nseg) return;
    const int64_t nr = *nruns;
    const int64_t a = lower_bound_u64(uniq, nr, sg[s].base), b = lower_bound_u64(uniq, nr, sg[s].base + cells[s]);
    fc[2 * s] = a;
    fc[2 * s + 1] = b - a;
}

__global__ void k_loop_gather(const float4* __restrict__ pts, const GatherEntry* __restrict__ ent, float4* __restrict__ dst0, float4* __restrict__ dst1) {
    const GatherEntry e = ent[blockIdx.x];
    float4* __restrict__ d = (e.which ? dst1 : dst0) + e.dst;
    for (int64_t i = threadIdx.x; i < e.count; i += blockDim.x) {
        const float4 p = __ldg(pts + e.src + i);
        d[i] = make_float4(p.x, p.y, p.z, 0.0f);
    }
}

// ---- extractSurroundingKeyFrames: the keyframe list of the local map
constexpr unsigned long long kNone = ~0ull;
struct SurrHdr {    // device header of the selection, read back with the list
    int64_t n_list, n_kept, err, pad;
    int32_t mm[6];  // key-pose min / max (ordered ints)
    int32_t stop;   // highest j <= cur with time_cur - time_j >= 10.0, -1 when none
    int32_t pad2;
};

// k_loop_detect's squared distance (FLANN L2_Simple<float>)
__device__ __forceinline__ float kf_d2(float qx, float qy, float qz, const KfRec& r) {
    const float dx = __fsub_rn(qx, r.T[3]), dy = __fsub_rn(qy, r.T[7]), dz = __fsub_rn(qz, r.T[11]);
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}
__device__ __forceinline__ int ordered_int(float f) {
    const int a = __float_as_int(f);
    return a >= 0 ? a : a ^ 0x7fffffff;
}
__device__ __forceinline__ float from_ordered(int a) { return __int_as_float(a >= 0 ? a : a ^ 0x7fffffff); }

__global__ void k_surr_init(SurrHdr* hdr) {
    if (threadIdx.x != 0) return;
    hdr->n_list = 0; hdr->n_kept = 0; hdr->err = 0;
    for (int k = 0; k < 3; ++k) { hdr->mm[k] = INT_MAX; hdr->mm[3 + k] = INT_MIN; }
    hdr->stop = -1;
}
// radiusSearch(keyframe cur): key (d2 bits, j) for every j <= cur strictly inside r2, kNone otherwise; and the recent walk's stop
__global__ void k_surr_hits(const KfRec* __restrict__ rec, int64_t cur, float r2, double time_cur, unsigned long long* __restrict__ key, SurrHdr* hdr) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j > cur) return;
    const float d2 = kf_d2(rec[cur].T[3], rec[cur].T[7], rec[cur].T[11], rec[j]);
    key[j] = d2 < r2 ? ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned long long)j : kNone;
    if (!(time_cur - rec[j].time < 10.0)) atomicMax(&hdr->stop, (int)j);
}
// the hits' positions in (d2, j) order, and their min / max
__global__ void k_surr_pos(const KfRec* __restrict__ rec, const unsigned long long* __restrict__ sorted, int64_t n, float4* __restrict__ pos, SurrHdr* hdr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || sorted[i] == kNone) return;
    const KfRec& r = rec[sorted[i] & 0xffffffffull];
    const float v[3] = {r.T[3], r.T[7], r.T[11]};
    pos[i] = make_float4(v[0], v[1], v[2], 0.0f);
    for (int k = 0; k < 3; ++k) {
        atomicMin(&hdr->mm[k], ordered_int(v[k]));
        atomicMax(&hdr->mm[3 + k], ordered_int(v[k]));
    }
}
// the key-pose VoxelGrid's leaf keys: vox::grid_from_minmax restated on the device (every thread derives the same grid), then
// vox::k_keys' arithmetic; kNone for the misses and when the grid is out of range (reported in hdr->err)
__global__ void k_surr_keys(const unsigned long long* __restrict__ sorted, const float4* __restrict__ pos, int64_t n, float inv_leaf, SurrHdr* hdr,
                            unsigned long long* __restrict__ keys, int32_t* __restrict__ vals) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    long long min_b[3] = {0, 0, 0}, div_b[3] = {1, 1, 1};
    bool ok = from_ordered(hdr->mm[0]) <= from_ordered(hdr->mm[3]);  // no hit: no grid
    unsigned long long c = 1;
    for (int k = 0; k < 3 && ok; ++k) {
        const float lo = floorf(__fmul_rn(from_ordered(hdr->mm[k]), inv_leaf)), hi = floorf(__fmul_rn(from_ordered(hdr->mm[3 + k]), inv_leaf));
        bool in = fabsf(lo) < 4.0e18f && fabsf(hi) < 4.0e18f;
        if (in) {
            min_b[k] = (long long)lo;
            div_b[k] = (long long)hi - min_b[k] + 1;
            const unsigned long long d = (unsigned long long)div_b[k];
            in = __umul64hi(c, d) == 0 && c * d <= 9000000000000000000ull;
            c *= d;
        }
        if (!in) {
            ok = false;
            if (i == 0) hdr->err = B200_ERR_RANGE;
        }
    }
    unsigned long long key = kNone;
    if (ok && sorted[i] != kNone) {
        const float4 p = pos[i];
        const long long i0 = (long long)(floorf(p.x * inv_leaf) - (float)min_b[0]);
        const long long i1 = (long long)(floorf(p.y * inv_leaf) - (float)min_b[1]);
        const long long i2 = (long long)(floorf(p.z * inv_leaf) - (float)min_b[2]);
        key = (unsigned long long)(i0 + i1 * div_b[0] + i2 * div_b[0] * div_b[1]);
    }
    keys[i] = key;
    vals[i] = (int32_t)i;
}
// one warp per key-pose centroid: its nearest keyframe among 0 .. cur (lexicographic minimum of (d2 bits, j): ties to the lower
// index), and whether the centroid passes extractCloud's gate sqrtf(d2 to keyframe cur) <= radius
__global__ void k_surr_nearest(const KfRec* __restrict__ rec, int64_t cur, const float4* __restrict__ cent, const unsigned long long* __restrict__ uniq,
                               const int32_t* __restrict__ nruns, float radius, int64_t* __restrict__ kf, uint8_t* __restrict__ pass) {
    const int lane = threadIdx.x & 31, nw = (int)((gridDim.x * (int64_t)blockDim.x) >> 5);
    const int nr = *nruns;
    for (int w = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5); w < nr; w += nw) {
        if (uniq[w] == kNone) continue;
        const float4 c = cent[w];
        unsigned long long best = kNone;
        for (int64_t j = lane; j <= cur; j += 32)
            best = min(best, ((unsigned long long)__float_as_uint(kf_d2(c.x, c.y, c.z, rec[j])) << 32) | (unsigned long long)j);
        for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
        if (lane == 0) {
            kf[w] = (int64_t)(best & 0xffffffffull);
            pass[w] = !(sqrtf(kf_d2(c.x, c.y, c.z, rec[cur])) > radius);
        }
    }
}
// the list in extraction order (centroids, then keyframes cur, cur-1, .. above the recent walk's stop), compacted through the
// distance gate; one block
__global__ void __launch_bounds__(1024) k_surr_list(const KfRec* __restrict__ rec, int64_t cur, const unsigned long long* __restrict__ uniq,
                                                    const int32_t* __restrict__ nruns, const int64_t* __restrict__ kf, const uint8_t* __restrict__ pass,
                                                    float radius, SurrHdr* hdr, int64_t* __restrict__ list) {
    using Scan = cub::BlockScan<int, 1024>;
    __shared__ typename Scan::TempStorage tmp;
    __shared__ int64_t base;
    const int nr = *nruns;
    const int64_t nc = nr - (nr > 0 && uniq[nr - 1] == kNone ? 1 : 0), nrec = cur - hdr->stop, total = nc + nrec;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (int64_t e0 = 0; e0 < total; e0 += 1024) {
        const int64_t e = e0 + threadIdx.x;
        int64_t k = -1;
        int ok = 0;
        if (e < nc) {
            k = kf[e];
            ok = pass[e];
        } else if (e < total) {
            k = cur - (e - nc);
            ok = !(sqrtf(kf_d2(rec[k].T[3], rec[k].T[7], rec[k].T[11], rec[cur])) > radius);
        }
        int at = 0, sum = 0;
        Scan(tmp).ExclusiveSum(ok, at, sum);
        if (ok) list[base + at] = k;
        __syncthreads();
        if (threadIdx.x == 0) base += sum;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        hdr->n_list = total;
        hdr->n_kept = base;
    }
}

}  // namespace loop
}  // namespace b200

using namespace b200;
using namespace b200::loop;

struct b200_keyframes : loop::SegWork {
    int device = 0;
    cudaStream_t stream = nullptr;
    float4* d_pool = nullptr;  // keyframe clouds end to end; grows by doubling
    int64_t pool_cap = 0, pool_used = 0;
    DevBuf<KfRec> d_rec;
    std::vector<KfRec> rec;     // host mirror of d_rec
    std::vector<int64_t> off, n;
    std::vector<int64_t> n_corner;  // corner points at the head of each cloud (b200_keyframes_add_features); -1: no split
    PinnedBuf<float4> h_stage;
    PinnedBuf<KfRec> h_rec;
    // detection and submap scratch (the rest is SegWork's)
    DevBuf<float4> d_raw;
    DevBuf<unsigned long long> d_cells;
    // local-map selection scratch
    DevBuf<float4> d_kpos;
    DevBuf<int64_t> d_sel;
    DevBuf<uint8_t> d_pass, d_hdr;
    PinnedBuf<uint8_t> h_sel;

    int64_t count() const { return (int64_t)n.size(); }
    void destroy() {
        cudaSetDevice(device);
        if (stream) cudaStreamSynchronize(stream);
        if (d_pool) cudaFree(d_pool);
        d_rec.release(); h_stage.release(); h_rec.release(); h_tab.release(); d_tab.release(); d_io.release(); h_io.release();
        d_raw.release(); d_cent.release(); d_mm.release(); h_mm.release(); k_in.release(); k_out.release(); k_uniq.release(); d_cells.release();
        v_in.release(); v_out.release(); run_cnt.release(); run_off.release(); d_cnt.release(); d_small.release(); keep.release(); cub_tmp.release();
        d_kpos.release(); d_sel.release(); d_pass.release(); d_hdr.release(); h_sel.release();
        if (stream) cudaStreamDestroy(stream);
    }
};

namespace b200 {
namespace loop {

int32_t check_params(const b200_loop_params* prm) {
    if (!prm) B200_FAIL(B200_ERR_ARG, "null loop parameters");
    if (!(prm->leaf > 0.f) || !std::isfinite(prm->leaf)) B200_FAIL(B200_ERR_ARG, "leaf must be positive");
    if (!(prm->search_radius >= 0.f) || prm->search_num < 0 || prm->min_source_points < 0 || prm->min_target_points < 0 || std::isnan(prm->time_gap))
        B200_FAIL(B200_ERR_ARG, "bad loop parameters");
    return B200_OK;
}
int32_t check_keys(const b200_keyframes* h, const int64_t* keys, int64_t n, bool allow_none) {
    for (int64_t i = 0; i < n; ++i)
        if (keys[i] >= h->count() || keys[i] < (allow_none ? -1 : 0)) B200_FAIL(B200_ERR_ARG, "keyframe index out of range");
    return B200_OK;
}
int32_t device_of(const b200_keyframes* h) { return h->device; }
int64_t raw_size(const b200_keyframes* h, int64_t key, int32_t num) {
    const int64_t lo = std::max<int64_t>(0, key - num), hi = std::min<int64_t>(h->count() - 1, key + num);
    return hi < lo ? 0 : h->off[hi] + h->n[hi] - h->off[lo];
}

int32_t detect(b200_keyframes* h, cudaStream_t s, const int64_t* cur, int64_t Q, const b200_loop_params& prm, int64_t* pre, float* sqdist) {
    CUDA_TRY(h->h_io.reserve(3 * (size_t)Q));
    CUDA_TRY(h->d_io.reserve(3 * (size_t)Q));
    memcpy(h->h_io.p, cur, Q * sizeof(int64_t));
    CUDA_TRY(cudaMemcpyAsync(h->d_io.p, h->h_io.p, Q * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    const float r2 = (float)((double)prm.search_radius * (double)prm.search_radius);  // pcl::KdTreeFLANN::radiusSearch: float(radius * radius)
    int64_t* d_pre = h->d_io.p + Q;
    float* d_sq = (float*)(h->d_io.p + 2 * Q);
    k_loop_detect<<<(unsigned)((Q * 32 + 255) / 256), 256, 0, s>>>(h->d_rec.p, h->d_io.p, (int)Q, r2, prm.time_gap, d_pre, d_sq);
    LAUNCH_COUNT(1);
    CUDA_TRY(cudaMemcpyAsync(h->h_io.p + Q, d_pre, 2 * Q * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
    memcpy(pre, h->h_io.p + Q, Q * sizeof(int64_t));
    if (sqdist) memcpy(sqdist, h->h_io.p + 2 * Q, Q * sizeof(float));
    return B200_OK;
}

void near_parts(const b200_keyframes* h, int64_t key, int32_t num, std::vector<Part>& parts) {
    const int64_t lo = std::max<int64_t>(0, key - num), hi = std::min<int64_t>(h->count() - 1, key + num);
    for (int64_t k = lo; k <= hi; ++k) parts.push_back(Part{k, 0, h->n[k]});
}

int32_t submaps(b200_keyframes* h, cudaStream_t s, const Seg* segs, int64_t nseg, int64_t group, float leaf, Submaps& out) {
    std::vector<Part> parts;
    std::vector<int64_t> part_off(1, 0);
    for (int64_t j = 0; j < nseg; ++j) {
        near_parts(h, segs[j].key, segs[j].num, parts);
        part_off.push_back((int64_t)parts.size());
    }
    const std::vector<float> leaves(nseg, leaf);
    return assemble(h, s, parts.data(), part_off.data(), leaves.data(), nseg, group, out);
}

int32_t assemble(b200_keyframes* h, cudaStream_t s, const Part* parts, const int64_t* part_off, const float* leaf, int64_t nseg, int64_t group,
                 Submaps& out) {
    // the (segment, part) table and the raw segment offsets, one upload
    std::vector<int64_t> off(nseg + 1, 0);
    std::vector<AsmEntry> ent;
    for (int64_t j = 0; j < nseg; ++j) {
        int64_t at = off[j];
        for (int64_t p = part_off[j]; p < part_off[j + 1]; ++p) {
            const Part& q = parts[p];
            if (q.count > 0) ent.push_back(AsmEntry{q.kf, h->off[q.kf] + q.begin, q.count, at});
            at += q.count;
        }
        off[j + 1] = at;
    }
    const size_t off_bytes = (nseg + 1) * sizeof(int64_t), seg_bytes = nseg * sizeof(SegGrid) + nseg * sizeof(unsigned long long);
    const size_t tab_bytes = std::max(off_bytes + ent.size() * sizeof(AsmEntry), off_bytes + seg_bytes);
    CUDA_TRY(h->h_tab.reserve(tab_bytes));
    CUDA_TRY(h->d_tab.reserve(tab_bytes));
    memcpy(h->h_tab.p, off.data(), off_bytes);
    memcpy(h->h_tab.p + off_bytes, ent.data(), ent.size() * sizeof(AsmEntry));
    CUDA_TRY(cudaMemcpyAsync(h->d_tab.p, h->h_tab.p, off_bytes + ent.size() * sizeof(AsmEntry), cudaMemcpyHostToDevice, s));
    const int64_t* d_off = (const int64_t*)h->d_tab.p;
    const int64_t nraw = off[nseg];
    CUDA_TRY(h->d_raw.reserve(std::max<int64_t>(nraw, 1)));
    if (!ent.empty()) {
        k_loop_assemble<<<(unsigned)ent.size(), 256, 0, s>>>(h->d_pool, h->d_rec.p, (const AsmEntry*)(h->d_tab.p + off_bytes), h->d_raw.p);
        LAUNCH_COUNT(1);
    }
    return seg_downsample(*h, s, h->d_raw.p, d_off, off.data(), off_bytes, leaf, nseg, group, out);
}

int32_t seg_downsample(SegWork& w, cudaStream_t s, const float4* pts, const int64_t* d_off, const int64_t* off, size_t grid_at, const float* leaf,
                       int64_t nseg, int64_t group, Submaps& out) {
    const size_t off_bytes = grid_at;
    CUDA_TRY(w.h_tab.reserve(grid_at + nseg * (sizeof(SegGrid) + sizeof(unsigned long long))));
    CUDA_TRY(w.d_tab.reserve(grid_at + nseg * (sizeof(SegGrid) + sizeof(unsigned long long))));
    // per-segment min / max, read back once
    int64_t max_n = 1;
    for (int64_t j = 0; j < nseg; ++j) max_n = std::max(max_n, off[j + 1] - off[j]);
    CUDA_TRY(w.d_mm.reserve(6 * (size_t)nseg));
    CUDA_TRY(w.h_mm.reserve(6 * (size_t)nseg));
    ndt::k_ndt_minmax_init<<<(unsigned)((6 * nseg + 255) / 256), 256, 0, s>>>(w.d_mm.p, (int)nseg);
    ndt::k_ndt_minmax<<<dim3((unsigned)std::min<int64_t>((max_n + 1023) / 1024, 256), (unsigned)nseg), 256, 0, s>>>(pts, d_off, w.d_mm.p);
    LAUNCH_COUNT(2);
    CUDA_TRY(cudaMemcpyAsync(w.h_mm.p, w.d_mm.p, 6 * nseg * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
    // every segment's grid as b200_voxel_downsample derives it; the cell ranges end to end
    out.status.assign(nseg, B200_OK);
    out.first.assign(nseg, 0);
    out.count.assign(nseg, 0);
    std::vector<SegGrid> sg(nseg);
    std::vector<unsigned long long> cells(nseg, 0);
    constexpr unsigned long long kMaxCells = 9000000000000000000ull;  // b200_voxel_downsample's bound for one cloud
    unsigned long long total = 0;
    int64_t done = 0;
    while (done < nseg) {
        unsigned long long gc = 0;
        for (int64_t j = done; j < done + group; ++j) {
            vox::Grid g{};
            SegGrid& q = sg[j];
            memset(&q, 0, sizeof q);
            const std::string err = g_last_error;
            out.status[j] = vox::grid_from_minmax(w.h_mm.p + 6 * j, leaf[j], g, cells[j]);
            if (out.status[j]) { g_last_error = err; cells[j] = 0; continue; }  // reported in the segment's status
            for (int k = 0; k < 3; ++k) { q.min_b[k] = g.min_b[k]; q.div_b[k] = g.div_b[k]; }
            q.inv_leaf = 1.0f / leaf[j];
            q.live = cells[j] > 0;
            gc += cells[j];
        }
        if (done > 0 && total + gc > kMaxCells) break;  // the next chunk takes it
        for (int64_t j = done; j < done + group; ++j) { sg[j].base = total; total += cells[j]; }
        done += group;
    }
    out.done = done;
    const int64_t n = off[done];
    if (n == 0) return B200_OK;
    const unsigned long long sentinel = total;
    int end_bit = 1;
    while (end_bit < 64 && (1ull << end_bit) <= sentinel) ++end_bit;
    // the grids replace the keyframe table (consumed by k_loop_assemble, which precedes on the stream)
    CUDA_TRY(cudaStreamSynchronize(s));
    memcpy(w.h_tab.p + off_bytes, sg.data(), done * sizeof(SegGrid));
    memcpy(w.h_tab.p + off_bytes + done * sizeof(SegGrid), cells.data(), done * sizeof(unsigned long long));
    CUDA_TRY(cudaMemcpyAsync(w.d_tab.p + off_bytes, w.h_tab.p + off_bytes, done * (sizeof(SegGrid) + sizeof(unsigned long long)), cudaMemcpyHostToDevice, s));
    const SegGrid* d_sg = (const SegGrid*)(w.d_tab.p + off_bytes);
    const unsigned long long* d_cells = (const unsigned long long*)(w.d_tab.p + off_bytes + done * sizeof(SegGrid));
    CUDA_TRY(w.k_in.reserve(n)); CUDA_TRY(w.k_out.reserve(n)); CUDA_TRY(w.k_uniq.reserve(n));
    CUDA_TRY(w.v_in.reserve(n)); CUDA_TRY(w.v_out.reserve(n)); CUDA_TRY(w.run_cnt.reserve(n)); CUDA_TRY(w.run_off.reserve(n));
    CUDA_TRY(w.d_cent.reserve(n)); CUDA_TRY(w.d_cnt.reserve(n)); CUDA_TRY(w.keep.reserve(n)); CUDA_TRY(w.d_small.reserve(4));
    CUDA_TRY(w.d_io.reserve(2 * (size_t)done)); CUDA_TRY(w.h_io.reserve(2 * (size_t)done));
    k_loop_keys<<<dim3((unsigned)std::min<int64_t>((max_n + 255) / 256, 1024), (unsigned)done), 256, 0, s>>>(pts, d_off, d_sg, sentinel, w.k_in.p,
                                                                                                          w.v_in.p);
    int32_t* d_nruns = w.d_small.p;
    size_t t1 = 0, t2 = 0, t3 = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, t1, w.k_in.p, w.k_out.p, w.v_in.p, w.v_out.p, (int)n, 0, end_bit, s));
    CUDA_TRY(cub::DeviceRunLengthEncode::Encode(nullptr, t2, w.k_out.p, w.k_uniq.p, w.run_cnt.p, d_nruns, (int)n, s));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, t3, w.run_cnt.p, w.run_off.p, (int)n, s));
    const size_t tmp = std::max(t1, std::max(t2, t3));
    CUDA_TRY(w.cub_tmp.reserve(tmp));
    size_t tt = tmp;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(w.cub_tmp.p, tt, w.k_in.p, w.k_out.p, w.v_in.p, w.v_out.p, (int)n, 0, end_bit, s));
    tt = tmp;
    CUDA_TRY(cub::DeviceRunLengthEncode::Encode(w.cub_tmp.p, tt, w.k_out.p, w.k_uniq.p, w.run_cnt.p, d_nruns, (int)n, s));
    tt = tmp;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(w.cub_tmp.p, tt, w.run_cnt.p, w.run_off.p, (int)n, s));
    const unsigned nb = (unsigned)((n + 255) / 256);
    vox::k_centroids<<<nb, 256, 0, s>>>(pts, w.v_out.p, w.k_uniq.p, w.run_off.p, w.run_cnt.p, d_nruns, sentinel, 0, w.d_cent.p, w.d_cnt.p,
                                        w.keep.p);
    k_loop_seg_runs<<<(unsigned)((done + 255) / 256), 256, 0, s>>>(w.k_uniq.p, d_nruns, d_sg, d_cells, (int)done, w.d_io.p);
    LAUNCH_COUNT(3);
    CUDA_TRY(cudaMemcpyAsync(w.h_io.p, w.d_io.p, 2 * done * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
    for (int64_t j = 0; j < done; ++j) {
        out.first[j] = w.h_io.p[2 * j];
        out.count[j] = w.h_io.p[2 * j + 1];
    }
    out.pts = w.d_cent.p;
    return B200_OK;
}

int32_t gather(b200_keyframes* h, cudaStream_t s, const float4* pts, const GatherEntry* e, int64_t n, float4* dst0, float4* dst1) {
    if (n < 1) return B200_OK;
    CUDA_TRY(h->h_tab.reserve(n * sizeof(GatherEntry)));
    CUDA_TRY(h->d_tab.reserve(n * sizeof(GatherEntry)));
    memcpy(h->h_tab.p, e, n * sizeof(GatherEntry));
    CUDA_TRY(cudaMemcpyAsync(h->d_tab.p, h->h_tab.p, n * sizeof(GatherEntry), cudaMemcpyHostToDevice, s));
    k_loop_gather<<<(unsigned)n, 256, 0, s>>>(pts, (const GatherEntry*)h->d_tab.p, dst0, dst1);
    LAUNCH_COUNT(1);
    CUDA_TRY(cudaGetLastError());
    return B200_OK;
}

cudaStream_t stream_of(const b200_keyframes* h) { return h->stream; }

int32_t check_surround(const b200_keyframes* h, int64_t cur, double time_cur, const b200_surround_params* prm) {
    if (!h || !prm) B200_FAIL(B200_ERR_ARG, "bad argument");
    const auto pos = [](float v) { return v > 0.f && std::isfinite(v); };
    if (!pos(prm->search_radius) || !pos(prm->density) || !pos(prm->corner_leaf) || !pos(prm->surf_leaf) || std::isnan(time_cur))
        B200_FAIL(B200_ERR_ARG, "bad surrounding-keyframe parameters");
    if (cur < -1 || cur >= std::max<int64_t>(h->count(), 1)) B200_FAIL(B200_ERR_ARG, "keyframe index out of range");
    return B200_OK;
}

int32_t surrounding(b200_keyframes* h, int64_t cur, double time_cur, const b200_surround_params& prm, Surround& out) {
    if (h->count() == 0) return B200_NO_EFFECTIVE_POINTS;  // extractSurroundingKeyFrames returns early on an empty cloudKeyPoses3D
    if (cur < 0) cur = h->count() - 1;
    cudaStream_t s = h->stream;
    const int64_t n = cur + 1;
    constexpr int64_t kListHead = 4096;  // list entries read back with the header; a longer list takes a second copy
    CUDA_TRY(h->d_hdr.reserve(sizeof(SurrHdr)));
    CUDA_TRY(h->d_sel.reserve(n + 2 * n));
    CUDA_TRY(h->h_sel.reserve(sizeof(SurrHdr) + kListHead * sizeof(int64_t)));
    CUDA_TRY(h->d_pass.reserve(n));
    CUDA_TRY(h->d_kpos.reserve(2 * n));
    CUDA_TRY(h->k_in.reserve(n)); CUDA_TRY(h->k_out.reserve(n)); CUDA_TRY(h->k_uniq.reserve(n));
    CUDA_TRY(h->v_in.reserve(n)); CUDA_TRY(h->v_out.reserve(n)); CUDA_TRY(h->run_cnt.reserve(n)); CUDA_TRY(h->run_off.reserve(n));
    CUDA_TRY(h->d_cnt.reserve(n)); CUDA_TRY(h->keep.reserve(n)); CUDA_TRY(h->d_small.reserve(4));
    SurrHdr* hdr = (SurrHdr*)h->d_hdr.p;
    int64_t* d_kf = h->d_sel.p;       // nearest keyframe of each centroid
    int64_t* d_list = h->d_sel.p + n;  // the list after the gate (at most n centroids + n recent keyframes)
    float4* pos = h->d_kpos.p;         // hit positions in (d2, j) order, then the centroids
    int32_t* d_nruns = h->d_small.p;
    const float r2 = (float)((double)prm.search_radius * (double)prm.search_radius);  // pcl::KdTreeFLANN::radiusSearch
    const unsigned nb = (unsigned)((n + 255) / 256);
    k_surr_init<<<1, 32, 0, s>>>(hdr);
    k_surr_hits<<<nb, 256, 0, s>>>(h->d_rec.p, cur, r2, time_cur, h->k_in.p, hdr);
    size_t t1 = 0, t2 = 0, t3 = 0, t4 = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortKeys(nullptr, t1, h->k_in.p, h->k_out.p, (int)n, 0, 64, s));
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, t2, h->k_in.p, h->k_uniq.p, h->v_in.p, h->v_out.p, (int)n, 0, 64, s));
    CUDA_TRY(cub::DeviceRunLengthEncode::Encode(nullptr, t3, h->k_uniq.p, h->k_in.p, h->run_cnt.p, d_nruns, (int)n, s));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, t4, h->run_cnt.p, h->run_off.p, (int)n, s));
    const size_t tmp = std::max(std::max(t1, t2), std::max(t3, t4));
    CUDA_TRY(h->cub_tmp.reserve(tmp));
    size_t tt = tmp;
    // hits first, in ascending (d2, j)
    CUDA_TRY(cub::DeviceRadixSort::SortKeys(h->cub_tmp.p, tt, h->k_in.p, h->k_out.p, (int)n, 0, 64, s));
    k_surr_pos<<<nb, 256, 0, s>>>(h->d_rec.p, h->k_out.p, n, pos, hdr);
    k_surr_keys<<<nb, 256, 0, s>>>(h->k_out.p, pos, n, 1.0f / prm.density, hdr, h->k_in.p, h->v_in.p);
    // the key-pose VoxelGrid: stable sort by leaf, runs, k_centroids (fp32 sums in (d2, j) order)
    tt = tmp;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(h->cub_tmp.p, tt, h->k_in.p, h->k_uniq.p, h->v_in.p, h->v_out.p, (int)n, 0, 64, s));
    tt = tmp;
    CUDA_TRY(cub::DeviceRunLengthEncode::Encode(h->cub_tmp.p, tt, h->k_uniq.p, h->k_in.p, h->run_cnt.p, d_nruns, (int)n, s));
    tt = tmp;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(h->cub_tmp.p, tt, h->run_cnt.p, h->run_off.p, (int)n, s));
    vox::k_centroids<<<nb, 256, 0, s>>>(pos, h->v_out.p, h->k_in.p, h->run_off.p, h->run_cnt.p, d_nruns, kNone, 0, pos + n, h->d_cnt.p, h->keep.p);
    k_surr_nearest<<<(unsigned)std::min<int64_t>((n + 7) / 8, 148 * 8), 256, 0, s>>>(h->d_rec.p, cur, pos + n, h->k_in.p, d_nruns, prm.search_radius,
                                                                                     d_kf, h->d_pass.p);
    k_surr_list<<<1, 1024, 0, s>>>(h->d_rec.p, cur, h->k_in.p, d_nruns, d_kf, h->d_pass.p, prm.search_radius, hdr, d_list);
    LAUNCH_COUNT(7);
    // read-back 1: the header and the head of the list
    CUDA_TRY(cudaMemcpyAsync(h->h_sel.p, hdr, sizeof(SurrHdr), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(h->h_sel.p + sizeof(SurrHdr), d_list, (size_t)std::min<int64_t>(2 * n, kListHead) * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
    const SurrHdr hh = *(const SurrHdr*)h->h_sel.p;
    if (hh.err) B200_FAIL((int32_t)hh.err, "density too small for the key-pose extent");
    out.n_list = hh.n_list;
    out.keys.resize(hh.n_kept);
    if (hh.n_kept > kListHead) {
        CUDA_TRY(cudaMemcpyAsync(out.keys.data(), d_list, (size_t)hh.n_kept * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
    } else if (hh.n_kept > 0) {
        memcpy(out.keys.data(), h->h_sel.p + sizeof(SurrHdr), (size_t)hh.n_kept * sizeof(int64_t));
    }
    // extractCloud: corner cloud -> segment 0, surf cloud -> segment 1, a keyframe listed twice appended twice
    std::vector<Part> parts;
    parts.reserve(2 * out.keys.size());
    out.raw[0] = out.raw[1] = 0;
    for (int pass = 0; pass < 2; ++pass)
        for (const int64_t k : out.keys) {
            const int64_t nc = h->n_corner[k];
            if (nc < 0) B200_FAIL(B200_ERR_ARG, "keyframe without a corner / surf split (added with b200_keyframes_add)");
            const Part p = pass == 0 ? Part{k, 0, nc} : Part{k, nc, h->n[k] - nc};
            parts.push_back(p);
            out.raw[pass] += p.count;
        }
    if (out.raw[0] + out.raw[1] > (int64_t)0x7fffff00) B200_FAIL(B200_ERR_ARG, "local map larger than 2^31 points");
    const int64_t part_off[3] = {0, (int64_t)out.keys.size(), 2 * (int64_t)out.keys.size()};
    const float leaves[2] = {prm.corner_leaf, prm.surf_leaf};
    if (const int32_t rc = assemble(h, s, parts.data(), part_off, leaves, 2, 2, out.sm)) return rc;
    for (int k = 0; k < 2; ++k)
        if (out.sm.status[k]) B200_FAIL(out.sm.status[k], "leaf size too small for the local map extent");
    return B200_OK;
}

}  // namespace loop
}  // namespace b200

extern "C" {

int32_t b200_keyframes_create(int32_t device, b200_keyframes** out) {
    if (!out) B200_FAIL(B200_ERR_ARG, "null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) B200_FAIL(B200_ERR_CUDA, "no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) B200_FAIL(B200_ERR_ARG, "bad device ordinal");
    b200_keyframes* h = new b200_keyframes();
    h->device = device;
    const auto init = [&]() -> int32_t {
        CUDA_SET_DEVICE(device);
        CUDA_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        return B200_OK;
    };
    const int32_t rc = init();
    if (rc) { h->destroy(); delete h; return rc; }
    *out = h;
    return B200_OK;
}
int32_t b200_keyframes_destroy(b200_keyframes* h) {
    if (!h) return B200_OK;
    h->destroy();
    delete h;
    return B200_OK;
}
int64_t b200_keyframes_count(b200_keyframes* h) { return h ? h->count() : -1; }

}  // extern "C"

// room for n more points in the pool
static int32_t pool_reserve(b200_keyframes* h, int64_t n) {
    cudaStream_t s = h->stream;
    if (h->pool_used + n > h->pool_cap) {  // double the pool, keep what it holds
        const int64_t cap = std::max<int64_t>(std::max<int64_t>(2 * h->pool_cap, h->pool_used + n), 1 << 20);
        float4* q = nullptr;
        CUDA_TRY(cudaMalloc(&q, (size_t)cap * sizeof(float4)));
        if (h->pool_used) {
            const cudaError_t e = cudaMemcpyAsync(q, h->d_pool, (size_t)h->pool_used * sizeof(float4), cudaMemcpyDeviceToDevice, s);
            if (e == cudaSuccess) cudaStreamSynchronize(s);
            if (e != cudaSuccess) { cudaFree(q); CUDA_TRY(e); }
        }
        if (h->d_pool) cudaFree(h->d_pool);
        h->d_pool = q;
        h->pool_cap = cap;
    }
    return B200_OK;
}

// appends one keyframe whose cloud is the concatenation of the nparts clouds src[i] (n[i] records at stride[i] bytes)
static int32_t keyframes_add(b200_keyframes* h, int nparts, const float* const* src, const int64_t* np, const int64_t* stride, const float* pose6,
                             double time, int64_t n_corner, int64_t* key) {
    int64_t n = 0;
    for (int i = 0; i < nparts; ++i) {
        if (np[i] < 0 || (np[i] > 0 && !src[i]) || stride[i] < 12) B200_FAIL(B200_ERR_ARG, "bad argument");
        n += np[i];
    }
    if (!h || !pose6 || n > (int64_t)0x7fffff00) B200_FAIL(B200_ERR_ARG, "bad argument");
    if (h->count() >= (int64_t)0x7fffffff) B200_FAIL(B200_ERR_ARG, "keyframe store full");
    CUDA_SET_DEVICE(h->device);
    cudaStream_t s = h->stream;
    const int64_t K = h->count();
    if (const int32_t rc = pool_reserve(h, n)) return rc;
    KfRec r;
    pose_matrix(pose6, r.T);
    r.time = time;
    CUDA_TRY(h->d_rec.reserve_keep((size_t)K + 1, (size_t)K, s));
    CUDA_TRY(h->h_stage.reserve((size_t)std::max<int64_t>(n, 1)));
    CUDA_TRY(h->h_rec.reserve(1));
    int64_t at = 0;
    for (int k = 0; k < nparts; ++k) {
        const char* c = (const char*)src[k];
        for (int64_t i = 0; i < np[k]; ++i) {
            const float* p = (const float*)(c + i * stride[k]);
            h->h_stage.p[at++] = make_float4(p[0], p[1], p[2], stride[k] >= 16 ? p[3] : 0.0f);
        }
    }
    h->h_rec.p[0] = r;
    if (n) CUDA_TRY(cudaMemcpyAsync(h->d_pool + h->pool_used, h->h_stage.p, (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(h->d_rec.p + K, h->h_rec.p, sizeof(KfRec), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    h->rec.push_back(r);
    h->off.push_back(h->pool_used);
    h->n.push_back(n);
    h->n_corner.push_back(n_corner);
    h->pool_used += n;
    if (key) *key = K;
    return B200_OK;
}

extern "C" {

int32_t b200_keyframes_add(b200_keyframes* h, const float* xyzi, int64_t n, int64_t stride, const float* pose6, double time, int64_t* key) {
    return keyframes_add(h, 1, &xyzi, &n, &stride, pose6, time, -1, key);
}

int32_t b200_keyframes_add_features(b200_keyframes* h, const float* corner, int64_t n_corner, int64_t stride_corner, const float* surf, int64_t n_surf,
                                    int64_t stride_surf, const float* pose6, double time, int64_t* key) {
    const float* src[2] = {corner, surf};
    const int64_t np[2] = {n_corner, n_surf}, stride[2] = {stride_corner, stride_surf};
    return keyframes_add(h, 2, src, np, stride, pose6, time, n_corner, key);
}

int32_t b200_keyframes_add_features_device(b200_keyframes* h, const void* d_corner, int64_t n_corner, const void* d_surf, int64_t n_surf,
                                           const float* pose6, double time, int64_t* key) {
    if (!h || !pose6 || n_corner < 0 || n_surf < 0 || n_corner + n_surf > (int64_t)0x7fffff00) B200_FAIL(B200_ERR_ARG, "bad argument");
    if (h->count() >= (int64_t)0x7fffffff) B200_FAIL(B200_ERR_ARG, "keyframe store full");
    CUDA_SET_DEVICE(h->device);
    if (const int32_t rc = check_device_buffer(d_corner, n_corner, h->device)) return rc;
    if (const int32_t rc = check_device_buffer(d_surf, n_surf, h->device)) return rc;
    cudaStream_t s = h->stream;
    const int64_t K = h->count(), n = n_corner + n_surf;
    if (const int32_t rc = pool_reserve(h, n)) return rc;
    KfRec r;
    pose_matrix(pose6, r.T);
    r.time = time;
    CUDA_TRY(h->d_rec.reserve_keep((size_t)K + 1, (size_t)K, s));
    CUDA_TRY(h->h_rec.reserve(1));
    h->h_rec.p[0] = r;
    if (n_corner) CUDA_TRY(cudaMemcpyAsync(h->d_pool + h->pool_used, d_corner, (size_t)n_corner * sizeof(float4), cudaMemcpyDeviceToDevice, s));
    if (n_surf) CUDA_TRY(cudaMemcpyAsync(h->d_pool + h->pool_used + n_corner, d_surf, (size_t)n_surf * sizeof(float4), cudaMemcpyDeviceToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(h->d_rec.p + K, h->h_rec.p, sizeof(KfRec), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    h->rec.push_back(r);
    h->off.push_back(h->pool_used);
    h->n.push_back(n);
    h->n_corner.push_back(n_corner);
    h->pool_used += n;
    if (key) *key = K;
    return B200_OK;
}

int32_t b200_keyframes_set_poses(b200_keyframes* h, int64_t first, int64_t count, const float* poses6) {
    if (!h || !poses6 || first < 0 || count < 1 || first + count > h->count()) B200_FAIL(B200_ERR_ARG, "bad argument");
    CUDA_SET_DEVICE(h->device);
    CUDA_TRY(h->h_rec.reserve((size_t)count));
    for (int64_t i = 0; i < count; ++i) {
        KfRec& r = h->rec[first + i];
        pose_matrix(poses6 + 6 * i, r.T);
        h->h_rec.p[i] = r;
    }
    CUDA_TRY(cudaMemcpyAsync(h->d_rec.p + first, h->h_rec.p, (size_t)count * sizeof(KfRec), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return B200_OK;
}

int32_t b200_loop_detect(b200_keyframes* h, const int64_t* cur, int64_t Q, const b200_loop_params* prm, int64_t* pre, float* sqdist) {
    if (!h || !cur || !prm || !pre || Q < 1 || Q > (int64_t)1 << 26) B200_FAIL(B200_ERR_ARG, "bad argument");
    if (const int32_t rc = check_params(prm)) return rc;
    if (const int32_t rc = check_keys(h, cur, Q, false)) return rc;
    CUDA_SET_DEVICE(h->device);
    return detect(h, h->stream, cur, Q, *prm, pre, sqdist);
}

int32_t b200_loop_submap(b200_keyframes* h, int64_t key, int32_t search_num, float leaf, float* out_xyzi, int64_t max_out, int64_t* n_out) {
    if (!h || !n_out || search_num < 0 || !(leaf > 0.f) || !std::isfinite(leaf) || max_out < 0 || (max_out > 0 && !out_xyzi))
        B200_FAIL(B200_ERR_ARG, "bad argument");
    if (const int32_t rc = check_keys(h, &key, 1, false)) return rc;
    if (raw_size(h, key, search_num) > (int64_t)0x7fffff00) B200_FAIL(B200_ERR_ARG, "submap larger than 2^31 points");
    CUDA_SET_DEVICE(h->device);
    const Seg seg{key, search_num};
    Submaps sm;
    const int32_t rc = submaps(h, h->stream, &seg, 1, 1, leaf, sm);
    if (rc) return rc;
    if (sm.status[0]) B200_FAIL(sm.status[0], "leaf size too small for the submap extent");
    *n_out = sm.count[0];
    const int64_t m = std::min(sm.count[0], max_out);
    if (m > 0) CUDA_TRY(cudaMemcpyAsync(out_xyzi, sm.pts + sm.first[0], (size_t)m * sizeof(float4), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return B200_OK;
}

int32_t b200_keyframes_surrounding(b200_keyframes* h, int64_t cur, double time_cur, const b200_surround_params* prm, int64_t* keys, int64_t max_keys,
                                   int64_t* n_keys) {
    if (!n_keys || max_keys < 0 || (max_keys > 0 && !keys)) B200_FAIL(B200_ERR_ARG, "bad argument");
    if (const int32_t rc = check_surround(h, cur, time_cur, prm)) return rc;
    CUDA_SET_DEVICE(h->device);
    Surround sr;
    *n_keys = 0;
    const int32_t rc = surrounding(h, cur, time_cur, *prm, sr);
    if (rc) return rc;
    *n_keys = (int64_t)sr.keys.size();
    std::copy(sr.keys.begin(), sr.keys.begin() + std::min<int64_t>(max_keys, (int64_t)sr.keys.size()), keys);
    return B200_OK;
}

int32_t b200_keyframes_surrounding_map(b200_keyframes* h, int64_t cur, double time_cur, const b200_surround_params* prm, float* corner_xyzi,
                                       int64_t max_corner, int64_t* n_corner, float* surf_xyzi, int64_t max_surf, int64_t* n_surf) {
    if (!n_corner || !n_surf || max_corner < 0 || max_surf < 0 || (max_corner > 0 && !corner_xyzi) || (max_surf > 0 && !surf_xyzi))
        B200_FAIL(B200_ERR_ARG, "bad argument");
    if (const int32_t rc = check_surround(h, cur, time_cur, prm)) return rc;
    CUDA_SET_DEVICE(h->device);
    Surround sr;
    *n_corner = *n_surf = 0;
    const int32_t rc = surrounding(h, cur, time_cur, *prm, sr);
    if (rc) return rc;
    *n_corner = sr.sm.count[0];
    *n_surf = sr.sm.count[1];
    float* dst[2] = {corner_xyzi, surf_xyzi};
    const int64_t cap[2] = {max_corner, max_surf};
    for (int k = 0; k < 2; ++k) {
        const int64_t m = std::min(sr.sm.count[k], cap[k]);
        if (m > 0) CUDA_TRY(cudaMemcpyAsync(dst[k], sr.sm.pts + sr.sm.first[k], (size_t)m * sizeof(float4), cudaMemcpyDeviceToHost, h->stream));
    }
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return B200_OK;
}

}  // extern "C"
