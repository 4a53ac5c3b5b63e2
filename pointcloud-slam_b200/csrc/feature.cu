// b200reg — the LOAM front end on the device: imageProjection's projection and cloud extraction, featureExtraction and
// mapOptimization's downsampleCurrentScan (LIO-SAM, from which jueying_slam derives), restated in oracle/feature_oracle.cpp.
//
// projection   one thread per input point: finite, range and ring tests, the column (velodyne / ouster: from the azimuth;
//              livox: the point's rank among the passing points of its line in input order, from one stable radix sort of
//              the line ids), then atomicMin of the input index on its pixel, so the first point of a pixel wins.
// extraction   one exclusive scan over the occupancy of the N_SCAN x Horizon_SCAN image gives every occupied pixel its
//              place in the extracted cloud (row-major, columns ascending) and every ring its start / end index.
// smoothness   one thread per index: curvature, the sort entry (curvature bits << 32 | index), occlusion and parallel-beam
//              marks (flags only ever set to 1), and the extent of the neighbour walk on each side (stops at a column jump
//              > 10), so that the greedy passes need no column reads.
// sorting      the sort ranges [sp, ep) of all regions of all rings are disjoint and their entries are fixed before step 5,
//              so one segmented sort orders all of them before the greedy passes.
// features     one warp per ring (rings never interact: S_{i+1} - E_i = 10), the six regions in order; a pass takes 32
//              sorted entries at a time, ballots the candidates and picks them lowest lane first; a pick's marks are one
//              contiguous index interval, which every lane applies to its own candidate without a memory round trip.
//              The ring's surf list is written into the ring's own index range, padded with NaN, so that every ring is one
//              segment of the segmented VoxelGrid (loop::seg_downsample, non-finite points skipped).
// downsample   the per-ring surf lists (one segment per ring, odometrySurfLeafSize) give surfaceCloud in ring order; then
//              cornerCloud and surfaceCloud (two segments) give the two DS clouds.
#include "common.cuh"
#include "loop.cuh"

#include <cub/cub.cuh>

#include <algorithm>
#include <cmath>
#include <vector>

namespace b200 {
namespace feat {

constexpr int kCornersPerRing = 20 * 6;
constexpr int32_t kEmpty = 0x7f7f7f7f;  // pixel owner after memset(0x7f): no point

struct Prm {
    int N, H, rate, livox;
    float min_r, max_r, edge, surf, ang_res;
};
struct Hdr {
    unsigned long long drop[4];  // non-finite, range, row, column
    unsigned long long passed;   // points that reached the pixel
};

__device__ __forceinline__ float range_of(float x, float y, float z) {
    return __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z)));
}

// tests of projectPointCloud up to the column; velodyne / ouster columns claim their pixel here, livox rows go to the sort
__global__ void k_feat_project(const uint8_t* __restrict__ in, int64_t n, int64_t stride, int ring_off, int ring_bytes, Prm p, Hdr* hdr,
                               uint32_t* __restrict__ row_key, int32_t* __restrict__ idx, int32_t* __restrict__ owner) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t* r = in + i * stride;
    const float x = *(const float*)r, y = *(const float*)(r + 4), z = *(const float*)(r + 8);
    uint32_t key = (uint32_t)p.N;
    if (p.livox) idx[i] = (int32_t)i;
    int drop = -1;
    if (!isfinite(x) || !isfinite(y) || !isfinite(z)) {
        drop = 0;
    } else {
        const float range = range_of(x, y, z);
        const int row = ring_bytes == 1 ? (int)r[ring_off] : (int)((unsigned)r[ring_off] | ((unsigned)r[ring_off + 1] << 8));
        if (range < p.min_r || range > p.max_r) drop = 1;
        else if (row >= p.N || row % p.rate != 0) drop = 2;
        else if (p.livox) key = (uint32_t)row;
        else {
            const float a = (float)atan2((double)x, (double)y);
            const float ha = (float)__ddiv_rn((double)__fmul_rn(a, 180.0f), M_PI);
            int col = (int)(-round(__ddiv_rn(__dsub_rn((double)ha, 90.0), (double)p.ang_res)) + (double)(p.H / 2));
            if (col >= p.H) col -= p.H;
            if (col < 0 || col >= p.H) drop = 3;
            else {
                atomicMin(owner + (int64_t)row * p.H + col, (int32_t)i);
                atomicAdd(&hdr->passed, 1ull);
            }
        }
    }
    if (drop >= 0) atomicAdd(&hdr->drop[drop], 1ull);
    if (p.livox) row_key[i] = key;
}

// livox: the column of a point is its rank within its line in input order (the keys are sorted stably)
__global__ void k_feat_livox(const uint32_t* __restrict__ key, const int32_t* __restrict__ idx, int64_t n, Prm p, Hdr* hdr, int32_t* __restrict__ owner) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const uint32_t row = key[q];
    if (row >= (uint32_t)p.N) return;
    int64_t lo = 0, hi = q;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (key[mid] < row) lo = mid + 1; else hi = mid;
    }
    const int64_t col = q - lo;
    if (col >= p.H) {
        atomicAdd(&hdr->drop[3], 1ull);
        return;
    }
    atomicMin(owner + (int64_t)row * p.H + col, idx[q]);
    atomicAdd(&hdr->passed, 1ull);
}

__global__ void k_feat_flags(const int32_t* __restrict__ owner, int64_t P, int32_t* __restrict__ flag) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q <= P) flag[q] = q < P && owner[q] != kEmpty ? 1 : 0;
}

// cloudExtraction: the occupied pixels in row-major order
__global__ void k_feat_extract(const uint8_t* __restrict__ in, int64_t stride, int64_t int_off, const int32_t* __restrict__ owner,
                               const int32_t* __restrict__ pos, int64_t P, int H, float4* __restrict__ cloud, int32_t* __restrict__ col,
                               float* __restrict__ range) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= P) return;
    const int32_t o = owner[q];
    if (o == kEmpty) return;
    const uint8_t* r = in + (int64_t)o * stride;
    const float x = *(const float*)r, y = *(const float*)(r + 4), z = *(const float*)(r + 8);
    const int32_t at = pos[q];
    cloud[at] = make_float4(x, y, z, int_off >= 0 ? *(const float*)(r + int_off) : 0.0f);
    col[at] = (int32_t)(q % H);
    range[at] = range_of(x, y, z);
}

// start / end ring indices, ring offsets and the sort ranges of the six regions of every ring
__global__ void k_feat_rings(const int32_t* __restrict__ pos, int N, int H, int32_t* __restrict__ start, int32_t* __restrict__ end,
                             int64_t* __restrict__ ring_off, int32_t* __restrict__ seg_b, int32_t* __restrict__ seg_e) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > N) return;
    ring_off[r] = pos[(int64_t)r * H];
    if (r == N) return;
    const int64_t S = (int64_t)pos[(int64_t)r * H] + 4, E = (int64_t)pos[(int64_t)(r + 1) * H] - 6;
    start[r] = (int32_t)S;
    end[r] = (int32_t)E;
    for (int j = 0; j < 6; ++j) {
        const int64_t sp = (S * (6 - j) + E * j) / 6, ep = (S * (5 - j) + E * (j + 1)) / 6 - 1;
        seg_b[6 * r + j] = sp < ep ? (int32_t)sp : 0;
        seg_e[6 * r + j] = sp < ep ? (int32_t)ep : 0;
    }
}

// calculateSmoothness and markOccludedPoints; fb[i] = forward walk length | backward walk length << 4 (0..5 each)
__global__ void k_feat_smooth(const float* __restrict__ r, const int32_t* __restrict__ col, const int32_t* __restrict__ d_m, int64_t cap,
                              unsigned long long* __restrict__ ent, uint8_t* __restrict__ fb, uint8_t* picked) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t m = *d_m;
    if (i >= m || i >= cap) return;
    float c = 0.0f;
    if (i >= 5 && i < m - 5) {
        float d = r[i - 5];
        d = __fadd_rn(d, r[i - 4]);
        d = __fadd_rn(d, r[i - 3]);
        d = __fadd_rn(d, r[i - 2]);
        d = __fadd_rn(d, r[i - 1]);
        d = __fsub_rn(d, __fmul_rn(r[i], 10.0f));
#pragma unroll
        for (int k = 1; k <= 5; ++k) d = __fadd_rn(d, r[i + k]);
        c = __fmul_rn(d, d);
    }
    ent[i] = ((unsigned long long)__float_as_uint(c) << 32) | (unsigned long long)i;
    int f = 0, b = 0;
    while (f < 5 && i + f + 1 < m && abs(col[i + f + 1] - col[i + f]) <= 10) ++f;
    while (b < 5 && i - b - 1 >= 0 && abs(col[i - b - 1] - col[i - b]) <= 10) ++b;
    fb[i] = (uint8_t)(f | (b << 4));
    if (i >= 5 && i < m - 6) {
        const float d1 = r[i], d2 = r[i + 1];
        if (abs(col[i + 1] - col[i]) < 10) {
            if ((double)__fsub_rn(d1, d2) > 0.3) {
                for (int k = 0; k <= 5; ++k) picked[i - k] = 1;
            } else if ((double)__fsub_rn(d2, d1) > 0.3) {
                for (int k = 1; k <= 6; ++k) picked[i + k] = 1;
            }
        }
        const double lim = __dmul_rn(0.02, (double)d1);
        if ((double)fabsf(__fsub_rn(r[i - 1], d1)) > lim && (double)fabsf(__fsub_rn(d2, d1)) > lim) picked[i] = 1;
    }
}

// extractFeatures for ring blockIdx.x, one warp
__global__ void __launch_bounds__(32) k_feat_pick(const unsigned long long* __restrict__ ent, const unsigned long long* __restrict__ sorted,
                                                  const uint8_t* __restrict__ fb, const float4* __restrict__ cloud, const int32_t* __restrict__ start,
                                                  const int32_t* __restrict__ end, const int64_t* __restrict__ ring_off, float edge, float surf,
                                                  uint8_t* picked, int8_t* label, float4* __restrict__ corner, int32_t* __restrict__ n_corner,
                                                  float4* __restrict__ surf_raw) {
    const int r = blockIdx.x, lane = threadIdx.x;
    const int64_t S = start[r], E = end[r];
    const int64_t base = ring_off[r], size = ring_off[r + 1] - base;
    const unsigned lt = (1u << lane) - 1u;
    int nc = 0;
    int64_t ns = 0;
    for (int j = 0; j < 6; ++j) {
        const int64_t sp = (S * (6 - j) + E * j) / 6, ep = (S * (5 - j) + E * (j + 1)) / 6 - 1;
        if (sp >= ep) continue;
        // corner pass, k = ep .. sp; the 21st candidate ends it
        int largest = 0;
        bool stop = false;
        for (int64_t hi = ep; hi >= sp && !stop; hi -= 32) {
            const int64_t k = hi - lane;
            bool cand = false;
            int64_t ind = 0;
            unsigned f = 0;
            if (k >= sp) {
                const unsigned long long e = k < ep ? sorted[k] : ent[ep];
                ind = (int64_t)(e & 0xffffffffull);
                cand = __uint_as_float((unsigned)(e >> 32)) > edge && picked[ind] == 0;
                f = fb[ind];
            }
            unsigned ball = __ballot_sync(~0u, cand);
            while (ball) {
                const int L = __ffs(ball) - 1;
                const int64_t pi = __shfl_sync(~0u, ind, L);
                const unsigned pf = __shfl_sync(~0u, f, L);
                if (++largest > 20) { stop = true; break; }
                const int fw = pf & 15, bw = pf >> 4;
                if (lane == 0) {
                    label[pi] = 1;
                    corner[(int64_t)r * kCornersPerRing + nc] = cloud[pi];
                }
                ++nc;
                if (lane <= fw + bw) picked[pi - bw + lane] = 1;
                if (ind >= pi - bw && ind <= pi + fw) cand = false;
                ball = __ballot_sync(~0u, cand);
            }
            __syncwarp();
        }
        // surf pass, k = sp .. ep
        for (int64_t lo = sp; lo <= ep; lo += 32) {
            const int64_t k = lo + lane;
            bool cand = false;
            int64_t ind = 0;
            unsigned f = 0;
            if (k <= ep) {
                const unsigned long long e = k < ep ? sorted[k] : ent[ep];
                ind = (int64_t)(e & 0xffffffffull);
                cand = __uint_as_float((unsigned)(e >> 32)) < surf && picked[ind] == 0;
                f = fb[ind];
            }
            unsigned ball = __ballot_sync(~0u, cand);
            while (ball) {
                const int L = __ffs(ball) - 1;
                const int64_t pi = __shfl_sync(~0u, ind, L);
                const unsigned pf = __shfl_sync(~0u, f, L);
                const int fw = pf & 15, bw = pf >> 4;
                if (lane == 0) label[pi] = -1;
                if (lane <= fw + bw) picked[pi - bw + lane] = 1;
                if (ind >= pi - bw && ind <= pi + fw) cand = false;
                ball = __ballot_sync(~0u, cand);
            }
            __syncwarp();
        }
        // the region's points with label <= 0, by index, into the ring's surf list
        for (int64_t lo = sp; lo <= ep; lo += 32) {
            const int64_t k = lo + lane;
            const bool take = k <= ep && label[k] <= 0;
            const unsigned ball = __ballot_sync(~0u, take);
            if (take) surf_raw[base + ns + __popc(ball & lt)] = cloud[k];
            ns += __popc(ball);
        }
        __syncwarp();
    }
    const float nan = __int_as_float(0x7fc00000);
    for (int64_t k = ns + lane; k < size; k += 32) surf_raw[base + k] = make_float4(nan, nan, nan, nan);
    if (lane == 0) n_corner[r] = nc;
}

// cornerCloud: the corners of ring blockIdx.x after those of the rings before it
__global__ void k_feat_corners(const float4* __restrict__ slots, const int32_t* __restrict__ n_corner, float4* __restrict__ out) {
    __shared__ int before;
    if (threadIdx.x == 0) before = 0;
    __syncthreads();
    int s = 0;
    for (int q = threadIdx.x; q < (int)blockIdx.x; q += blockDim.x) s += n_corner[q];
    atomicAdd(&before, s);
    __syncthreads();
    const int nc = n_corner[blockIdx.x];
    if ((int)threadIdx.x < nc) out[before + threadIdx.x] = slots[(int64_t)blockIdx.x * kCornersPerRing + threadIdx.x];
}

}  // namespace feat
}  // namespace b200

using namespace b200;
using namespace b200::feat;

struct b200_features {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    b200_feature_params prm{};
    Prm kp{};
    int64_t P = 0;  // pixels
    loop::SegWork w;
    DevBuf<uint8_t> d_in, d_fb, d_picked, cub_tmp;
    DevBuf<int8_t> d_label;
    DevBuf<uint32_t> d_key, d_key2;
    DevBuf<int32_t> d_idx, d_idx2, d_owner, d_flag, d_pos, d_col, d_start, d_end, d_seg, d_ncorner;
    DevBuf<float> d_range;
    DevBuf<unsigned long long> d_ent, d_sorted;
    DevBuf<float4> d_cloud, d_slots, d_surf_raw, d_cat, d_ds;
    DevBuf<int64_t> d_ring_off, d_off2;
    DevBuf<Hdr> d_hdr;
    PinnedBuf<Hdr> h_hdr;
    PinnedBuf<int64_t> h_ring_off, h_off2;
    PinnedBuf<int32_t> h_ncorner;
    // the last scan
    int64_t m = 0, n[4] = {0, 0, 0, 0};  // extracted; corner, surface, cornerDS, surfDS
    float4* dev[4] = {nullptr, nullptr, nullptr, nullptr};

    void release() {
        d_in.release(); d_fb.release(); d_picked.release(); cub_tmp.release(); d_label.release(); d_key.release(); d_key2.release();
        d_idx.release(); d_idx2.release(); d_owner.release(); d_flag.release(); d_pos.release(); d_col.release(); d_start.release(); d_end.release();
        d_seg.release(); d_ncorner.release(); d_range.release(); d_ent.release(); d_sorted.release(); d_cloud.release(); d_slots.release();
        d_surf_raw.release(); d_cat.release(); d_ds.release(); d_ring_off.release(); d_off2.release(); d_hdr.release(); h_hdr.release();
        h_ring_off.release(); h_off2.release(); h_ncorner.release();
        w.h_tab.release(); w.d_tab.release(); w.d_io.release(); w.h_io.release(); w.d_cent.release(); w.d_mm.release(); w.h_mm.release();
        w.k_in.release(); w.k_out.release(); w.k_uniq.release(); w.v_in.release(); w.v_out.release(); w.run_cnt.release(); w.run_off.release();
        w.d_cnt.release(); w.d_small.release(); w.keep.release(); w.cub_tmp.release();
    }
};

// VoxelGrid of device segments pts[off[j] .. off[j+1]) with leaf[j], results appended to dst in segment order; *n_out points.
// Segments are taken in as many seg_downsample calls as the 64-bit sort key needs.
static int32_t feat_downsample(b200_features* h, const float4* pts, const int64_t* off, const float* leaf, int64_t nseg, int64_t group, float4* dst,
                               int64_t* n_out, int64_t* per_seg) {
    cudaStream_t s = h->stream;
    CUDA_TRY(h->d_off2.reserve(nseg + 1));
    CUDA_TRY(h->h_off2.reserve(nseg + 1));
    int64_t d0 = 0, total = 0;
    while (d0 < nseg) {
        const int64_t k = nseg - d0;
        CUDA_TRY(cudaStreamSynchronize(s));  // h_off2 may still feed an earlier copy
        for (int64_t j = 0; j <= k; ++j) h->h_off2.p[j] = off[d0 + j] - off[d0];
        CUDA_TRY(cudaMemcpyAsync(h->d_off2.p, h->h_off2.p, (k + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
        loop::Submaps sm;
        if (const int32_t rc = loop::seg_downsample(h->w, s, pts + off[d0], h->d_off2.p, h->h_off2.p, 0, leaf + d0, k, group, sm)) return rc;
        for (int64_t j = 0; j < sm.done; ++j) {
            if (sm.status[j] != B200_OK) B200_FAIL(sm.status[j], "VoxelGrid of more than 9e18 leaves");
            if (per_seg) per_seg[d0 + j] = sm.count[j];
        }
        const int64_t got = sm.done ? sm.first[sm.done - 1] + sm.count[sm.done - 1] : 0;
        if (got) CUDA_TRY(cudaMemcpyAsync(dst + total, sm.pts, got * sizeof(float4), cudaMemcpyDeviceToDevice, s));
        total += got;
        d0 += sm.done;
    }
    *n_out = total;
    return B200_OK;
}

static int32_t feat_check(const b200_feature_params* p) {
    if (!p) B200_FAIL(B200_ERR_ARG, "null feature parameters");
    if (p->n_scan < 1 || p->n_scan > 1024 || p->horizon_scan < 1 || (int64_t)p->n_scan * p->horizon_scan > (1 << 26)) B200_FAIL(B200_ERR_ARG, "bad image size");
    if (p->downsample_rate < 1 || (p->sensor != 0 && p->sensor != 1)) B200_FAIL(B200_ERR_ARG, "bad downsampleRate or sensor");
    for (float leaf : {p->odometry_surf_leaf, p->mapping_corner_leaf, p->mapping_surf_leaf})
        if (!(leaf > 0.f) || !std::isfinite(leaf)) B200_FAIL(B200_ERR_ARG, "leaf sizes must be positive");
    if (std::isnan(p->min_range) || std::isnan(p->max_range) || std::isnan(p->edge_threshold) || std::isnan(p->surf_threshold))
        B200_FAIL(B200_ERR_ARG, "NaN parameter");
    return B200_OK;
}

extern "C" {

int32_t b200_features_create(const b200_feature_params* prm, int32_t device, b200_features** out) {
    if (!out) B200_FAIL(B200_ERR_ARG, "bad argument");
    if (const int32_t rc = feat_check(prm)) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) B200_FAIL(B200_ERR_CUDA, "no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) B200_FAIL(B200_ERR_ARG, "bad device ordinal");
    CUDA_SET_DEVICE(device);
    b200_features* h = new b200_features();
    h->device = device;
    h->prm = *prm;
    h->kp = Prm{prm->n_scan, prm->horizon_scan, prm->downsample_rate, prm->sensor, prm->min_range, prm->max_range, prm->edge_threshold,
                prm->surf_threshold, (float)(360.0 / (float)prm->horizon_scan)};
    h->P = (int64_t)prm->n_scan * prm->horizon_scan;
    const int N = prm->n_scan;
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev1);
    if (e == cudaSuccess) e = h->d_owner.reserve(h->P);
    if (e == cudaSuccess) e = h->d_flag.reserve(h->P + 1);
    if (e == cudaSuccess) e = h->d_pos.reserve(h->P + 1);
    if (e == cudaSuccess) e = h->d_start.reserve(N);
    if (e == cudaSuccess) e = h->d_end.reserve(N);
    if (e == cudaSuccess) e = h->d_seg.reserve(12 * (size_t)N);
    if (e == cudaSuccess) e = h->d_ncorner.reserve(N);
    if (e == cudaSuccess) e = h->d_slots.reserve((size_t)N * kCornersPerRing);
    if (e == cudaSuccess) e = h->d_ring_off.reserve(N + 1);
    if (e == cudaSuccess) e = h->d_hdr.reserve(1);
    if (e == cudaSuccess) e = h->h_hdr.reserve(1);
    if (e == cudaSuccess) e = h->h_ring_off.reserve(N + 1);
    if (e == cudaSuccess) e = h->h_ncorner.reserve(N);
    if (e != cudaSuccess) {
        b200_features_destroy(h);
        B200_FAIL(B200_ERR_CUDA, cudaGetErrorString(e));
    }
    *out = h;
    return B200_OK;
}

int32_t b200_features_destroy(b200_features* h) {
    if (!h) return B200_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    h->release();
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return B200_OK;
}

int32_t b200_features_extract(b200_features* h, const void* points, int64_t n, int64_t stride, int64_t intensity_offset, int64_t ring_offset,
                              int32_t ring_bytes, b200_feature_info* info) {
    if (!h || n < 0 || (n && !points) || n > (int64_t)0x7f000000 || stride < 12 || stride % 4 || (ring_bytes != 1 && ring_bytes != 2) ||
        ring_offset < 0 || ring_offset + ring_bytes > stride || (intensity_offset >= 0 && (intensity_offset % 4 || intensity_offset + 4 > stride)))
        B200_FAIL(B200_ERR_ARG, "bad argument");
    CUDA_SET_DEVICE(h->device);
    cudaStream_t s = h->stream;
    const int N = h->prm.n_scan, H = h->prm.horizon_scan;
    const int64_t P = h->P, cap = std::max<int64_t>(std::min<int64_t>(n, P), 1);
    h->m = 0;
    for (int k = 0; k < 4; ++k) h->n[k] = 0;
    CUDA_TRY(h->d_in.reserve(std::max<int64_t>(n * stride, 1)));
    CUDA_TRY(h->d_key.reserve(std::max<int64_t>(n, 1))); CUDA_TRY(h->d_key2.reserve(std::max<int64_t>(n, 1)));
    CUDA_TRY(h->d_idx.reserve(std::max<int64_t>(n, 1))); CUDA_TRY(h->d_idx2.reserve(std::max<int64_t>(n, 1)));
    CUDA_TRY(h->d_cloud.reserve(cap)); CUDA_TRY(h->d_col.reserve(cap)); CUDA_TRY(h->d_range.reserve(cap));
    CUDA_TRY(h->d_ent.reserve(cap)); CUDA_TRY(h->d_sorted.reserve(cap)); CUDA_TRY(h->d_fb.reserve(cap));
    CUDA_TRY(h->d_picked.reserve(cap)); CUDA_TRY(h->d_label.reserve(cap)); CUDA_TRY(h->d_surf_raw.reserve(cap));
    CUDA_TRY(h->d_cat.reserve(cap + (int64_t)N * kCornersPerRing)); CUDA_TRY(h->d_ds.reserve(cap + (int64_t)N * kCornersPerRing));
    CUDA_TRY(cudaEventRecord(h->ev0, s));
    if (n) CUDA_TRY(cudaMemcpyAsync(h->d_in.p, points, n * stride, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemsetAsync(h->d_hdr.p, 0, sizeof(Hdr), s));
    CUDA_TRY(cudaMemsetAsync(h->d_owner.p, 0x7f, P * sizeof(int32_t), s));
    CUDA_TRY(cudaMemsetAsync(h->d_picked.p, 0, cap, s));
    CUDA_TRY(cudaMemsetAsync(h->d_label.p, 0, cap, s));
    const Prm& kp = h->kp;
    const unsigned nb = (unsigned)std::max<int64_t>((n + 255) / 256, 1);
    k_feat_project<<<nb, 256, 0, s>>>(h->d_in.p, n, stride, (int)ring_offset, ring_bytes, kp, h->d_hdr.p, h->d_key.p, h->d_idx.p, h->d_owner.p);
    LAUNCH_COUNT(1);
    if (kp.livox && n) {
        size_t t = 0;
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, t, h->d_key.p, h->d_key2.p, h->d_idx.p, h->d_idx2.p, (int)n, 0, 32, s));
        CUDA_TRY(h->cub_tmp.reserve(t));
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(h->cub_tmp.p, t, h->d_key.p, h->d_key2.p, h->d_idx.p, h->d_idx2.p, (int)n, 0, 32, s));
        k_feat_livox<<<nb, 256, 0, s>>>(h->d_key2.p, h->d_idx2.p, n, kp, h->d_hdr.p, h->d_owner.p);
        LAUNCH_COUNT(2);
    }
    const unsigned pb = (unsigned)((P + 1 + 255) / 256);
    k_feat_flags<<<pb, 256, 0, s>>>(h->d_owner.p, P, h->d_flag.p);
    size_t t = 0;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, t, h->d_flag.p, h->d_pos.p, (int)(P + 1), s));
    size_t t2 = 0;
    CUDA_TRY(cub::DeviceSegmentedSort::SortKeys(nullptr, t2, h->d_ent.p, h->d_sorted.p, (int)cap, 6 * N, h->d_seg.p, h->d_seg.p + 6 * N, s));
    CUDA_TRY(h->cub_tmp.reserve(std::max(t, t2)));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(h->cub_tmp.p, t, h->d_flag.p, h->d_pos.p, (int)(P + 1), s));
    k_feat_extract<<<(unsigned)((P + 255) / 256), 256, 0, s>>>(h->d_in.p, stride, intensity_offset, h->d_owner.p, h->d_pos.p, P, H, h->d_cloud.p,
                                                              h->d_col.p, h->d_range.p);
    k_feat_rings<<<(unsigned)((N + 1 + 127) / 128), 128, 0, s>>>(h->d_pos.p, N, H, h->d_start.p, h->d_end.p, h->d_ring_off.p, h->d_seg.p,
                                                                 h->d_seg.p + 6 * N);
    const int32_t* d_m = h->d_pos.p + P;
    k_feat_smooth<<<(unsigned)((cap + 255) / 256), 256, 0, s>>>(h->d_range.p, h->d_col.p, d_m, cap, h->d_ent.p, h->d_fb.p, h->d_picked.p);
    t2 = h->cub_tmp.cap;
    CUDA_TRY(cub::DeviceSegmentedSort::SortKeys(h->cub_tmp.p, t2, h->d_ent.p, h->d_sorted.p, (int)cap, 6 * N, h->d_seg.p, h->d_seg.p + 6 * N, s));
    k_feat_pick<<<N, 32, 0, s>>>(h->d_ent.p, h->d_sorted.p, h->d_fb.p, h->d_cloud.p, h->d_start.p, h->d_end.p, h->d_ring_off.p, kp.edge, kp.surf,
                                 h->d_picked.p, h->d_label.p, h->d_slots.p, h->d_ncorner.p, h->d_surf_raw.p);
    k_feat_corners<<<N, kCornersPerRing, 0, s>>>(h->d_slots.p, h->d_ncorner.p, h->d_cat.p);
    LAUNCH_COUNT(9);
    // the one read-back of the counts
    CUDA_TRY(cudaMemcpyAsync(h->h_hdr.p, h->d_hdr.p, sizeof(Hdr), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(h->h_ring_off.p, h->d_ring_off.p, (N + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(h->h_ncorner.p, h->d_ncorner.p, N * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
    const Hdr hd = *h->h_hdr.p;
    const int64_t m = h->h_ring_off.p[N];
    int64_t nc = 0;
    for (int r = 0; r < N; ++r) nc += h->h_ncorner.p[r];
    h->m = m;
    int32_t rc = B200_OK;
    int64_t ns = 0, ncd = 0, nsd = 0;
    if (m == 0) {
        rc = B200_NO_EFFECTIVE_POINTS;
    } else {
        // surfaceCloud: one segment per ring, written after cornerCloud
        std::vector<float> leaves((size_t)std::max(N, 2), h->prm.odometry_surf_leaf);
        rc = feat_downsample(h, h->d_surf_raw.p, h->h_ring_off.p, leaves.data(), N, 1, h->d_cat.p + nc, &ns, nullptr);
        if (rc == B200_OK) {
            // downsampleCurrentScan: cornerCloud and surfaceCloud as two segments
            const int64_t off3[3] = {0, nc, nc + ns};
            const float leaf2[2] = {h->prm.mapping_corner_leaf, h->prm.mapping_surf_leaf};
            int64_t per[2] = {0, 0}, nds = 0;
            rc = feat_downsample(h, h->d_cat.p, off3, leaf2, 2, 2, h->d_ds.p, &nds, per);
            ncd = per[0];
            nsd = per[1];
        }
    }
    CUDA_TRY(cudaEventRecord(h->ev1, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h->ev0, h->ev1);
    if (rc == B200_OK) {
        h->n[0] = nc; h->n[1] = ns; h->n[2] = ncd; h->n[3] = nsd;
    }
    h->dev[0] = h->d_cat.p; h->dev[1] = h->d_cat.p + h->n[0]; h->dev[2] = h->d_ds.p; h->dev[3] = h->d_ds.p + h->n[2];
    if (info) {
        info->n_in = n;
        for (int k = 0; k < 4; ++k) (&info->dropped_nonfinite)[k] = (int64_t)hd.drop[k];
        info->dropped_dup = (int64_t)hd.passed - m;
        info->n_extracted = m;
        info->n_corner = h->n[0]; info->n_surface = h->n[1]; info->n_corner_ds = h->n[2]; info->n_surf_ds = h->n[3];
        info->gpu_ms = ms;
    }
    if (rc < 0) h->m = 0;
    return rc;
}

int32_t b200_features_cloud_info(b200_features* h, float* cloud_xyzi, int32_t* col, float* range, int32_t* start_ring, int32_t* end_ring, int64_t max,
                                 int64_t* n) {
    if (!h || !n || max < 0) B200_FAIL(B200_ERR_ARG, "bad argument");
    CUDA_SET_DEVICE(h->device);
    *n = h->m;
    const int64_t k = std::min(max, h->m);
    cudaStream_t s = h->stream;
    if (cloud_xyzi && k) CUDA_TRY(cudaMemcpyAsync(cloud_xyzi, h->d_cloud.p, k * sizeof(float4), cudaMemcpyDeviceToHost, s));
    if (col && k) CUDA_TRY(cudaMemcpyAsync(col, h->d_col.p, k * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (range && k) CUDA_TRY(cudaMemcpyAsync(range, h->d_range.p, k * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (start_ring) CUDA_TRY(cudaMemcpyAsync(start_ring, h->d_start.p, h->prm.n_scan * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (end_ring) CUDA_TRY(cudaMemcpyAsync(end_ring, h->d_end.p, h->prm.n_scan * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return B200_OK;
}

int32_t b200_features_labels(b200_features* h, float* curvature, int8_t* label, uint8_t* picked, int64_t max, int64_t* n) {
    if (!h || !n || max < 0) B200_FAIL(B200_ERR_ARG, "bad argument");
    CUDA_SET_DEVICE(h->device);
    *n = h->m;
    const int64_t k = std::min(max, h->m);
    cudaStream_t s = h->stream;
    if (curvature && k) {
        std::vector<unsigned long long> e((size_t)k);
        CUDA_TRY(cudaMemcpyAsync(e.data(), h->d_ent.p, k * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        for (int64_t i = 0; i < k; ++i) {
            const uint32_t b = (uint32_t)(e[i] >> 32);
            memcpy(curvature + i, &b, 4);
        }
    }
    if (label && k) CUDA_TRY(cudaMemcpyAsync(label, h->d_label.p, k, cudaMemcpyDeviceToHost, s));
    if (picked && k) CUDA_TRY(cudaMemcpyAsync(picked, h->d_picked.p, k, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return B200_OK;
}

int32_t b200_features_cloud(b200_features* h, int32_t which, float* out_xyzi, int64_t max, int64_t* n) {
    if (!h || !n || which < 0 || which > 3 || max < 0 || (max && !out_xyzi)) B200_FAIL(B200_ERR_ARG, "bad argument");
    CUDA_SET_DEVICE(h->device);
    *n = h->n[which];
    const int64_t k = std::min(max, h->n[which]);
    if (k) CUDA_TRY(cudaMemcpyAsync(out_xyzi, h->dev[which], k * sizeof(float4), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return B200_OK;
}

const void* b200_features_device_cloud(b200_features* h, int32_t which, int64_t* n) {
    if (!h || which < 0 || which > 3) return nullptr;
    if (n) *n = h->n[which];
    return h->dev[which];
}

int32_t b200_features_device(b200_features* h) { return h ? h->device : -1; }

}  // extern "C"
