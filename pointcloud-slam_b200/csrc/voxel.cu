// b200reg — voxel-grid reductions: scan downsample (pcl::VoxelGrid) and the keyframe-merge map builder.
//
// Replaces
//   pcl::VoxelGrid<PointType>::filter as jueying_lio calls it on every scan (jueying_lio/src/laser_mapping.cc:323-328,
//   leaf = filter_size_surf); PCL is third-party, its applyFilter is vendored nearly verbatim in
//   jueying_slam/include/voxel_grid_large.cpp:25-258 (min/max -> leaf index -> sort -> per-leaf centroid);
//   dynamic_map/construct_full_map <poses.txt> <frames_dir> <out.pcd> <leaf> (scripts/construct_full_map.sh:6) — sources
//   absent from the reference (SURVEY.md F3); built here as "move every keyframe by its pose, merge, VoxelGrid(leaf)".
//
// downsample   min/max -> 64-bit leaf index per point -> stable radix sort -> run-length segments -> one thread per
//              leaf sums x, y, z, intensity in fp32 in input order and divides by the count (the arithmetic of
//              pcl::CentroidPoint) -> centroids in ascending leaf-index order.  The result can stay on the device and feed
//              b200_iekf_update_device directly.
// map builder  a voxel hash table in HBM, one 32-byte record per voxel {key, count, fp32 sums of the offsets from the voxel corner
//              and of the intensity}; every keyframe is transformed (fp32,
//              pcl::transformPointCloud order) and accumulated with atomics, so keyframes stream through in any order
//              and any number per launch.  Across GPUs (one process each, keyframes split in contiguous blocks) the
//              partial sums are exchanged by voxel ownership (hash of the key) with grouped ncclSend/ncclRecv and merged;
//              afterwards every rank owns a disjoint part of the map.
#include "common.cuh"

#include <cub/cub.cuh>
#include <chrono>

#include <algorithm>
#include <cmath>
#include <vector>

#include "comm.cuh"

namespace b200 {
namespace vox {

__device__ __forceinline__ int f2ord(float f) {
    int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}

__global__ void k_minmax_init(int* mm) {
    if (threadIdx.x < 3) mm[threadIdx.x] = 0x7fffffff;
    else if (threadIdx.x < 6) mm[threadIdx.x] = (int)0x80000000;
}
__global__ void k_minmax(const float4* __restrict__ pts, int64_t n, int* __restrict__ mm) {
    float mn[3] = {3.402823466e+38f, 3.402823466e+38f, 3.402823466e+38f}, mx[3] = {-3.402823466e+38f, -3.402823466e+38f, -3.402823466e+38f};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 p = __ldg(pts + i);
        if (!(isfinite(p.x) && isfinite(p.y) && isfinite(p.z))) continue;
        mn[0] = fminf(mn[0], p.x); mn[1] = fminf(mn[1], p.y); mn[2] = fminf(mn[2], p.z);
        mx[0] = fmaxf(mx[0], p.x); mx[1] = fmaxf(mx[1], p.y); mx[2] = fmaxf(mx[2], p.z);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k)
        for (int o = 16; o > 0; o >>= 1) {
            mn[k] = fminf(mn[k], __shfl_xor_sync(0xffffffffu, mn[k], o));
            mx[k] = fmaxf(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
        }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            atomicMin(mm + k, f2ord(mn[k]));
            atomicMax(mm + 3 + k, f2ord(mx[k]));
        }
    }
}

struct Grid {
    long long min_b[3], div_b[3];
    float inv_leaf;
};

// leaf index of every point (voxel_grid_large.cpp:163-168), 64-bit; non-finite points get the sentinel and sort last
__global__ void k_keys(const float4* __restrict__ pts, int n, Grid g, unsigned long long sentinel, unsigned long long* __restrict__ keys,
                       int32_t* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = __ldg(pts + i);
    unsigned long long key = sentinel;
    if (isfinite(p.x) && isfinite(p.y) && isfinite(p.z)) {
        const long long i0 = (long long)(floorf(p.x * g.inv_leaf) - (float)g.min_b[0]);
        const long long i1 = (long long)(floorf(p.y * g.inv_leaf) - (float)g.min_b[1]);
        const long long i2 = (long long)(floorf(p.z * g.inv_leaf) - (float)g.min_b[2]);
        key = (unsigned long long)(i0 + i1 * g.div_b[0] + i2 * g.div_b[0] * g.div_b[1]);
    }
    keys[i] = key;
    vals[i] = i;
}

// one thread per leaf: fp32 sums in input order, divided by the count (pcl::CentroidPoint); compacts on min_points
__global__ void k_centroids(const float4* __restrict__ pts, const int32_t* __restrict__ sorted_idx, const unsigned long long* __restrict__ uniq,
                            const int32_t* __restrict__ run_off, const int32_t* __restrict__ run_cnt, const int32_t* __restrict__ nruns,
                            unsigned long long sentinel, int min_points, float4* __restrict__ out, int32_t* __restrict__ out_cnt,
                            uint8_t* __restrict__ keep) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= *nruns) return;
    const int c = run_cnt[r];
    const bool ok = uniq[r] != sentinel && c >= min_points;
    keep[r] = ok ? 1 : 0;
    out_cnt[r] = c;
    if (!ok) return;
    const int off = run_off[r];
    float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
    for (int k = 0; k < c; ++k) {
        const float4 p = __ldg(pts + __ldg(sorted_idx + off + k));
        sx += p.x; sy += p.y; sz += p.z; si += p.w;
    }
    const float n = (float)c;
    out[r] = make_float4(sx / n, sy / n, sz / n, si / n);
}

// ------------------------------------------------------------------ per-point motion compensation
// ImuProcess::UndistortPcl, backward half (jueying_lio/include/imu_processing.hpp:247-284): every point is moved from
// the sensor pose at its own sampling time to the pose at the end of the scan, using the IMU poses of the forward
// propagation (which stays on the host: a few dozen sequential esekf::predict calls).  fp64 like the reference.
struct ImuPose {  // common::Pose6D (common_lib.h:111-123)
    double t, acc[3], gyr[3], vel[3], pos[3], rot[9];
};
static_assert(sizeof(ImuPose) == 22 * 8, "22 doubles per pose");

__device__ inline void und_cross(const double* a, const double* b, double* r) {
    r[0] = a[1] * b[2] - a[2] * b[1];
    r[1] = a[2] * b[0] - a[0] * b[2];
    r[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ inline void und_qrot(const double* q /*x y z w*/, const double* v, double* r) {  // Eigen _transformVector
    double uv[3], c2[3];
    und_cross(q, v, uv);
    uv[0] += uv[0]; uv[1] += uv[1]; uv[2] += uv[2];
    und_cross(q, uv, c2);
    for (int i = 0; i < 3; ++i) r[i] = v[i] + q[3] * uv[i] + c2[i];
}
// one compensation step of point p (float coordinates in / out) in segment (head, tail)
__device__ inline void und_step(const ImuPose& head, const ImuPose& tail, const double* xe, double t, float* p) {
    const double dt = t - head.t;
    const double* w = tail.gyr;
    const double n = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
    double E[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    if (n > 0.0000001) {  // Exp(ang_vel, dt), so3_math.h:31-49
        const double a[3] = {w[0] / n, w[1] / n, w[2] / n};
        const double K[9] = {0.0, -a[2], a[1], a[2], 0.0, -a[0], -a[1], a[0], 0.0};
        const double ang = n * dt, s = sin(ang), c1 = 1.0 - cos(ang);
        double cK[9], KK[9];
        for (int i = 0; i < 9; ++i) cK[i] = c1 * K[i];
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) KK[i * 3 + j] = cK[i * 3] * K[j] + cK[i * 3 + 1] * K[3 + j] + cK[i * 3 + 2] * K[6 + j];
        for (int i = 0; i < 9; ++i) E[i] = (E[i] + s * K[i]) + KK[i];
    }
    double Ri[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) Ri[i * 3 + j] = head.rot[i * 3] * E[j] + head.rot[i * 3 + 1] * E[3 + j] + head.rot[i * 3 + 2] * E[6 + j];
    const double Pi[3] = {p[0], p[1], p[2]};
    const double* offT = xe + 11;
    const double rot_c[4] = {-xe[3], -xe[4], -xe[5], xe[6]}, offR_c[4] = {-xe[7], -xe[8], -xe[9], xe[10]};
    double Tei[3], a[3], b[3], c[3], d[3], e[3];
    for (int i = 0; i < 3; ++i) Tei[i] = ((head.pos[i] + head.vel[i] * dt) + 0.5 * tail.acc[i] * dt * dt) - xe[i];
    und_qrot(xe + 7, Pi, a);
    for (int i = 0; i < 3; ++i) a[i] += offT[i];
    for (int i = 0; i < 3; ++i) b[i] = (Ri[i * 3] * a[0] + Ri[i * 3 + 1] * a[1] + Ri[i * 3 + 2] * a[2]) + Tei[i];
    und_qrot(rot_c, b, c);
    for (int i = 0; i < 3; ++i) d[i] = c[i] - offT[i];
    und_qrot(offR_c, d, e);
    p[0] = (float)e[0]; p[1] = (float)e[1]; p[2] = (float)e[2];
}

// raw records -> (time key, index); time as an order-preserving uint so that a stable radix sort = ascending time.
// -0.0 is keyed as +0.0: the two compare equal, so they tie and keep their input order like any other tie.
__global__ void k_und_keys(const float* __restrict__ raw, int n, int stride_f, int time_index, uint32_t* __restrict__ keys, int32_t* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t u = __float_as_uint(raw[(size_t)i * stride_f + time_index]);
    if (u == 0x80000000u) u = 0u;
    keys[i] = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    vals[i] = i;
}
__global__ void k_undistort(const float* __restrict__ raw, const int32_t* __restrict__ order, int n, int stride_f, int time_index, int intensity_index,
                            const ImuPose* __restrict__ poses, int K, const double* __restrict__ xe, float4* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* r = raw + (size_t)order[i] * stride_f;
    float p[3] = {r[0], r[1], r[2]};
    const double t = (double)r[time_index] / double(1000);
    if (K >= 2) {
        // segment = largest k <= K-2 whose head offset is before t (the reference walks the segments backwards)
        int lo = -1, hi = K - 1;  // poses[lo].t < t (or lo == -1), poses[hi].t >= t or hi == K-1
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (poses[mid].t < t) lo = mid; else hi = mid;
        }
        if (lo >= 0) {
            und_step(poses[lo], poses[lo + 1], xe, t, p);
            // the earliest point is compensated again by every earlier segment (imu_processing.hpp:279-281)
            if (i == 0)
                for (int k = lo - 1; k >= 0; --k) und_step(poses[k], poses[k + 1], xe, t, p);
        }
    }
    out[i] = make_float4(p[0], p[1], p[2], intensity_index >= 0 ? r[intensity_index] : 0.0f);
}

// ------------------------------------------------------------------ map builder
struct __align__(16) Xfer {  // what travels between ranks: 32 bytes per voxel
    unsigned long long key;
    unsigned int n, pad;
    float4 s;  // sums of (x, y, z) - voxel corner and of the intensity, like Vox::s
};
static_assert(sizeof(Xfer) == 32, "exchange record");

__device__ __forceinline__ uint32_t mix64(unsigned long long k) {
    k ^= k >> 33;
    k *= 0xff51afd7ed558ccdULL;
    k ^= k >> 33;
    k *= 0xc4ceb9fe1a85ec53ULL;
    k ^= k >> 33;
    return (uint32_t)k;
}

// One voxel = ONE 32-byte record = one DRAM sector: key, count and the four sums.  The first layout kept key / fp64 sums / count
// in three arrays (three lines per point, 178 MB of DRAM traffic per 24-keyframe launch, ncu r01) and paid five atomics per
// point (four fp64 adds and the count).  Here a point costs TWO: one 16-byte vector atomic (red.global.add.v4.f32, sm_90+)
// and the count.  fp32 sums are exact enough because they are taken RELATIVE TO THE VOXEL'S CORNER: the offsets are below one
// leaf (0.1 m), so a voxel of a hundred points keeps its centroid to ~1e-8 m wherever the voxel sits (coordinates of a
// survey reach kilometres: absolute fp32 sums would be off by millimetres and depend on the order of the atomics).
// The corner is recovered from the key, so the offsets are rank independent and travel as they are.
struct __align__(32) Vox {
    unsigned long long key;
    unsigned int cnt, pad;
    float4 s;  // sum of (x - cx * leaf, y - cy * leaf, z - cz * leaf, intensity)
};
static_assert(sizeof(Vox) == 32, "voxel record");
struct Table {
    Vox* v;
    uint32_t mask;
};
__device__ __forceinline__ void unpack_cell(unsigned long long key, int& cx, int& cy, int& cz) {  // key = pack_key(cz, cy, cx)
    cx = (int)(key & 0x1FFFFFull) - kKeyBias;
    cy = (int)((key >> 21) & 0x1FFFFFull) - kKeyBias;
    cz = (int)((key >> 42) & 0x1FFFFFull) - kKeyBias;
}
// one point into its voxel: offset from the voxel corner (exact in fp64, then narrowed), one vector atomic + the count
__device__ __forceinline__ void vox_add(Vox* v, float x, float y, float z, float inten, int cx, int cy, int cz, double leaf) {
    const float4 d = make_float4((float)((double)x - (double)cx * leaf), (float)((double)y - (double)cy * leaf),
                                 (float)((double)z - (double)cz * leaf), inten);
    atomicAdd(&v->s, d);
    atomicAdd(&v->cnt, 1u);
}

// `created` counts the voxels this thread created; the caller adds the warp's total to the voxel counter with ONE atomic at
// the end of the kernel (count_created) - an atomicAdd per new voxel is millions of atomics on a single address.
__device__ __forceinline__ int table_slot(const Table& t, unsigned long long key, unsigned int& created, unsigned int* err) {
    uint32_t slot = mix64(key) & t.mask;
    for (uint32_t probes = 0; probes <= t.mask; ++probes) {
        const unsigned long long k = t.v[slot].key;
        if (k == key) return (int)slot;
        if (k == kEmptyKey) {
            const unsigned long long old = atomicCAS(&t.v[slot].key, kEmptyKey, key);
            if (old == kEmptyKey) {
                ++created;
                return (int)slot;
            }
            if (old == key) return (int)slot;
        }
        slot = (slot + 1) & t.mask;
    }
    atomicAdd(err, 1u);
    return -1;
}
// every thread of the block calls this once, converged, at the end of the kernel
__device__ __forceinline__ void count_created(unsigned int created, unsigned int* n_voxels, unsigned int capacity, unsigned int* err) {
    for (int o = 16; o > 0; o >>= 1) created += __shfl_xor_sync(0xffffffffu, created, o);
    if ((threadIdx.x & 31) == 0 && created) {
        if (atomicAdd(n_voxels, created) + created > capacity) atomicAdd(err, 1u);  // the table has >= 2 x capacity slots: flagged, not overrun
    }
}

// One keyframe (or several: `frame_of` maps a point to its pose) through pcl::transformPointCloud and into the table.
// Voxel cell = floor(p * inverse_leaf) per axis, exactly VoxelGrid's partition; the key orders voxels like VoxelGrid's
// leaf index does (z slowest, then y, then x).
struct PoseM {
    float m[12];  // row-major 3x4, travels as a kernel argument (no per-keyframe copy)
};
__global__ void k_accumulate(const float4* __restrict__ pts, int64_t n, PoseM pose, float inv_leaf, double leaf, Table t, unsigned int* n_voxels,
                             unsigned int capacity, unsigned int* err) {
    const float* M = pose.m;
    unsigned int created = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 p = __ldg(pts + i);
        const float x = ((M[0] * p.x + M[1] * p.y) + M[2] * p.z) + M[3];
        const float y = ((M[4] * p.x + M[5] * p.y) + M[6] * p.z) + M[7];
        const float z = ((M[8] * p.x + M[9] * p.y) + M[10] * p.z) + M[11];
        if (!(isfinite(x) && isfinite(y) && isfinite(z))) continue;
        const int cx = (int)floorf(x * inv_leaf), cy = (int)floorf(y * inv_leaf), cz = (int)floorf(z * inv_leaf);
        if (!cell_in_range(cx, cy, cz)) { atomicAdd(err + 1, 1u); continue; }
        const unsigned long long key = pack_key(cz, cy, cx);
        const int s = table_slot(t, key, created, err);
        if (s < 0) continue;
        vox_add(t.v + s, x, y, z, p.w, cx, cy, cz, leaf);
    }
    count_created(created, n_voxels, capacity, err);
}

// Several keyframes per launch (blockIdx.y = keyframe): one 100k-point keyframe is 391 blocks, less than three per SM, and
// its atomics and table probes are latency bound (ncu: 25 % of the warp slots active); a batch fills the machine.  The frame
// descriptors travel as a kernel argument (no per-batch copy).
constexpr int kFrameBatch = 24;
struct FrameDesc {
    const float4* pts;
    int64_t n;
    float m[12];
};
struct FrameBatch {
    FrameDesc f[kFrameBatch];
};
__global__ void __launch_bounds__(256) k_accumulate_batch(FrameBatch fb, float inv_leaf, double leaf, Table t, unsigned int* n_voxels, unsigned int capacity,
                                                          unsigned int* err) {
    const FrameDesc& d = fb.f[blockIdx.y];
    const float* M = d.m;
    const float4* __restrict__ pts = d.pts;
    const int64_t n = d.n;
    unsigned int created = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 p = __ldg(pts + i);
        const float x = ((M[0] * p.x + M[1] * p.y) + M[2] * p.z) + M[3];
        const float y = ((M[4] * p.x + M[5] * p.y) + M[6] * p.z) + M[7];
        const float z = ((M[8] * p.x + M[9] * p.y) + M[10] * p.z) + M[11];
        if (!(isfinite(x) && isfinite(y) && isfinite(z))) continue;
        const int cx = (int)floorf(x * inv_leaf), cy = (int)floorf(y * inv_leaf), cz = (int)floorf(z * inv_leaf);
        if (!cell_in_range(cx, cy, cz)) { atomicAdd(err + 1, 1u); continue; }
        const unsigned long long key = pack_key(cz, cy, cx);
        const int s = table_slot(t, key, created, err);
        if (s < 0) continue;
        vox_add(t.v + s, x, y, z, p.w, cx, cy, cz, leaf);
    }
    count_created(created, n_voxels, capacity, err);
}

__global__ void k_table_clear(Table t) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s > t.mask) return;
    Vox e{};
    e.key = kEmptyKey;
    t.v[s] = e;
}

// occupied slots -> (key, slot) pairs
__global__ void k_table_list(Table t, unsigned long long* __restrict__ keys, uint32_t* __restrict__ slots, unsigned int* n_out) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const unsigned long long k = s <= t.mask ? t.v[s].key : kEmptyKey;
    const unsigned live = __ballot_sync(0xffffffffu, k != kEmptyKey);  // one atomic per warp, not per voxel
    if (!live) return;
    const int leader = __ffs(live) - 1;
    unsigned int base = 0;
    if (lane == leader) base = atomicAdd(n_out, (unsigned int)__popc(live));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (k == kEmptyKey) return;
    const unsigned int i = base + (unsigned int)__popc(live & ((1u << lane) - 1u));
    keys[i] = k;
    slots[i] = s;
}

__global__ void k_extract(Table t, double leaf, const uint32_t* __restrict__ slots, int64_t m, float4* __restrict__ out, int32_t* __restrict__ out_cnt) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= m) return;
    const uint32_t s = slots[i];
    const Vox a = t.v[s];
    const double n = (double)a.cnt;
    int cx, cy, cz;
    unpack_cell(a.key, cx, cy, cz);
    out[i] = make_float4((float)((double)cx * leaf + (double)a.s.x / n), (float)((double)cy * leaf + (double)a.s.y / n),
                         (float)((double)cz * leaf + (double)a.s.z / n), (float)((double)a.s.w / n));
    if (out_cnt) out_cnt[i] = (int32_t)a.cnt;
}

// exchange: owner rank of a voxel, records grouped by owner
__device__ __forceinline__ int owner_of(unsigned long long key, int nranks) { return (int)((mix64(key ^ 0x9E3779B97F4A7C15ULL) >> 8) % (uint32_t)nranks); }

// Both kernels hand out positions per owner with ONE atomic per (warp, owner): a plain atomicAdd per voxel is millions of
// atomics on nranks addresses (2.3 ms for 4.4 M voxels on two ranks).
__global__ void k_owner_count(Table t, int nranks, unsigned long long* __restrict__ counts) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long k = s <= t.mask ? t.v[s].key : kEmptyKey;
    const int owner = k == kEmptyKey ? -1 : owner_of(k, nranks);
    const unsigned peers = __match_any_sync(0xffffffffu, owner);
    if (owner >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(counts + owner, (unsigned long long)__popc(peers));
}
__global__ void k_owner_scatter(Table t, int nranks, unsigned long long* __restrict__ cursor /*starts at the owner offsets*/, Xfer* __restrict__ out) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const unsigned long long k = s <= t.mask ? t.v[s].key : kEmptyKey;
    const int owner = k == kEmptyKey ? -1 : owner_of(k, nranks);
    const unsigned peers = __match_any_sync(0xffffffffu, owner);
    const int leader = __ffs(peers) - 1;
    unsigned long long base = 0;
    if (owner >= 0 && lane == leader) base = atomicAdd(cursor + owner, (unsigned long long)__popc(peers));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (owner < 0) return;
    const unsigned long long i = base + (unsigned long long)__popc(peers & ((1u << lane) - 1u));
    const Vox a = t.v[s];
    out[i] = Xfer{k, a.cnt, 0u, a.s};
}
__global__ void k_merge_records(const Xfer* __restrict__ rec, int64_t m, Table t, unsigned int* n_voxels, unsigned int capacity, unsigned int* err) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    unsigned int created = 0;
    if (i < m) {
        const Xfer r = rec[i];
        const int s = table_slot(t, r.key, created, err);
        if (s >= 0) {
            atomicAdd(&t.v[s].s, r.s);
            atomicAdd(&t.v[s].cnt, r.n);
        }
    }
    count_created(created, n_voxels, capacity, err);
}

static uint32_t next_pow2(uint64_t v) {
    uint32_t p = 1;
    while (p < v && p < (1u << 31)) p <<= 1;
    return p;
}

struct Builder {
    int device = 0;
    cudaStream_t stream = nullptr;
    float leaf = 0.1f, inv_leaf = 10.f;
    uint64_t capacity = 0;
    Table tab{}, tab2{};
    bool have_tab2 = false;
    unsigned int* d_ctr = nullptr;  // [0] voxels, [1] table errors, [2] range errors, [3] list count
    PinnedBuf<unsigned int> h_ctr;
    DevBuf<float4> d_pts, d_out;
    DevBuf<float> d_M;
    PinnedBuf<float> h_M;
    PinnedBuf<float4> h_stage;
    DevBuf<unsigned long long> d_keys, d_keys2, d_counts;
    DevBuf<uint32_t> d_slots, d_slots2;
    DevBuf<int32_t> d_cnt;
    DevBuf<uint8_t> cub_tmp;
    PinnedBuf<unsigned long long> h_counts;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int64_t frames = 0, points = 0;
    float ms_accumulate = 0.f, last_ms = 0.f;
    int64_t n_sorted = -1;  // entries of d_slots valid for extraction, -1 = stale
    static constexpr int NSTAGE = 3;
    PinnedBuf<float4> stage_h[NSTAGE];
    DevBuf<float4> stage_d[NSTAGE];
    cudaEvent_t stage_ev[NSTAGE] = {nullptr, nullptr, nullptr};
    int64_t host_frames = 0;

    int32_t alloc_table(Table& t) {
        const uint32_t T = next_pow2(2 * capacity);
        t.mask = T - 1;
        CUDA_TRY(cudaMalloc(&t.v, (size_t)T * sizeof(Vox)));
        k_table_clear<<<(T + 255) / 256, 256, 0, stream>>>(t);
        LAUNCH_COUNT(1);
        return B200_OK;
    }
    void free_table(Table& t) {
        cudaFree(t.v);
        t = Table{};
    }
    int32_t init(float leaf_, uint64_t cap, int dev) {
        if (!(leaf_ > 0.f) || cap < 1 || cap > (1ull << 30)) B200_FAIL(B200_ERR_ARG, "bad map-builder parameters");
        device = dev; leaf = leaf_; inv_leaf = 1.0f / leaf_; capacity = cap;
        CUDA_SET_DEVICE(dev);
        CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreate(&ev0));
        CUDA_TRY(cudaEventCreate(&ev1));
        CUDA_TRY(cudaMalloc(&d_ctr, 8 * sizeof(unsigned int)));
        CUDA_TRY(cudaMemsetAsync(d_ctr, 0, 8 * sizeof(unsigned int), stream));
        CUDA_TRY(h_ctr.reserve(8));
        CUDA_TRY(d_M.reserve(12));
        CUDA_TRY(h_M.reserve(12));
        int32_t rc = alloc_table(tab);
        if (rc) return rc;
        CUDA_TRY(cudaStreamSynchronize(stream));
        return B200_OK;
    }
    void destroy() {
        cudaSetDevice(device);
        if (stream) cudaStreamSynchronize(stream);
        free_table(tab);
        if (have_tab2) free_table(tab2);
        cudaFree(d_ctr);
        h_ctr.release(); d_pts.release(); d_out.release(); d_M.release(); h_M.release(); h_stage.release(); d_keys.release(); d_keys2.release();
        d_counts.release(); d_slots.release(); d_slots2.release(); d_cnt.release(); cub_tmp.release();
        h_counts.release();
        for (int i = 0; i < NSTAGE; ++i) { stage_h[i].release(); stage_d[i].release(); if (stage_ev[i]) cudaEventDestroy(stage_ev[i]); }
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (stream) cudaStreamDestroy(stream);
    }
    // T = Translation * Quaterniond in double, narrowed to float (poses.txt: x y z qw qx qy qz)
    static void pose_matrix(const double* p7, float* M) {
        const double w = p7[3], x = p7[4], y = p7[5], z = p7[6];
        const double R[9] = {1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                             2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                             2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)};
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) M[r * 4 + c] = (float)R[r * 3 + c];
            M[r * 4 + 3] = (float)p7[r];
        }
    }
    int32_t add_device(const float4* d_frame, int64_t n, const double* pose7) {
        CUDA_SET_DEVICE(device);
        PoseM pm;
        pose_matrix(pose7, pm.m);
        const int blocks = (int)std::min<int64_t>((n + 255) / 256, 148 * 8);
        k_accumulate<<<blocks, 256, 0, stream>>>(d_frame, n, pm, inv_leaf, (double)leaf, tab, d_ctr, (unsigned int)capacity, d_ctr + 1);
        LAUNCH_COUNT(1);
        ++frames;
        points += n;
        n_sorted = -1;
        return B200_OK;
    }
    int32_t add_device_batch(const void* const* d_frames, const int64_t* ns, const double* poses7, int64_t count) {
        CUDA_SET_DEVICE(device);
        for (int64_t c0 = 0; c0 < count; c0 += kFrameBatch) {
            const int k = (int)std::min<int64_t>(kFrameBatch, count - c0);
            FrameBatch fb{};
            int64_t nmax = 0;
            for (int j = 0; j < k; ++j) {
                fb.f[j].pts = (const float4*)d_frames[c0 + j];
                fb.f[j].n = ns[c0 + j];
                pose_matrix(poses7 + 7 * (c0 + j), fb.f[j].m);
                nmax = std::max(nmax, ns[c0 + j]);
                points += ns[c0 + j];
            }
            const int blocks = (int)std::min<int64_t>((nmax + 255) / 256, 148 * 8);
            k_accumulate_batch<<<dim3(blocks, k), 256, 0, stream>>>(fb, inv_leaf, (double)leaf, tab, d_ctr, (unsigned int)capacity, d_ctr + 1);
            LAUNCH_COUNT(1);
            frames += k;
        }
        n_sorted = -1;
        CUDA_TRY(cudaGetLastError());
        return B200_OK;
    }
    int32_t check() {
        CUDA_TRY(cudaMemcpyAsync(h_ctr.p, d_ctr, 8 * sizeof(unsigned int), cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        CUDA_TRY(cudaGetLastError());
        if (h_ctr.p[1]) B200_FAIL(B200_ERR_CAPACITY, "map builder: voxel capacity exceeded");
        if (h_ctr.p[2]) B200_FAIL(B200_ERR_RANGE, "map builder: point outside the voxel key range");
        return B200_OK;
    }
    // sorted list of the occupied slots (ascending key = VoxelGrid's leaf order)
    int32_t sort_slots() {
        int32_t rc = check();
        if (rc) return rc;
        const int64_t m = h_ctr.p[0];
        const uint32_t T = tab.mask + 1;
        CUDA_TRY(d_keys.reserve(m + 1)); CUDA_TRY(d_keys2.reserve(m + 1)); CUDA_TRY(d_slots.reserve(m + 1)); CUDA_TRY(d_slots2.reserve(m + 1));
        CUDA_TRY(cudaMemsetAsync(d_ctr + 3, 0, sizeof(unsigned int), stream));
        k_table_list<<<(T + 255) / 256, 256, 0, stream>>>(tab, d_keys.p, d_slots.p, d_ctr + 3);
        LAUNCH_COUNT(1);
        if (m > 0) {
            size_t tmp = 0;
            cub::DeviceRadixSort::SortPairs(nullptr, tmp, d_keys.p, d_keys2.p, d_slots.p, d_slots2.p, (int)m, 0, 63, stream);
            CUDA_TRY(cub_tmp.reserve(tmp));
            CUDA_TRY(cub::DeviceRadixSort::SortPairs(cub_tmp.p, tmp, d_keys.p, d_keys2.p, d_slots.p, d_slots2.p, (int)m, 0, 63, stream));
        }
        n_sorted = m;
        return B200_OK;
    }
};

}  // namespace vox
}  // namespace b200

using namespace b200;
struct b200_mapbuild { vox::Builder b; };
struct b200_downsampler {
    int device = 0;
    cudaStream_t stream = nullptr;
    DevBuf<float4> d_in, d_out, d_cmp;
    DevBuf<unsigned long long> k_in, k_out, k_uniq;
    DevBuf<int32_t> v_in, v_out, run_cnt, run_off, d_small, d_cnt, d_cnt_cmp;
    DevBuf<uint8_t> keep, cub_tmp;
    PinnedBuf<float4> h_stage;
    PinnedBuf<int32_t> h_small;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    float last_ms = 0.f;
    int64_t n_out = 0;
    // undistortion stage
    DevBuf<float> d_raw;
    DevBuf<uint32_t> u_keys_in, u_keys_out;
    DevBuf<int32_t> u_vals_in, u_vals_out;
    DevBuf<double> d_poses;
    PinnedBuf<double> h_poses;
    int64_t n_staged = 0;  // undistorted points waiting in d_in
};

static int32_t downsample_run(b200_downsampler* d, int64_t n, float leaf, int32_t min_points) {
    using namespace vox;
    cudaStream_t s = d->stream;
    CUDA_TRY(cudaEventRecord(d->ev0, s));
    int* mm = d->d_small.p;
    k_minmax_init<<<1, 32, 0, s>>>(mm);
    k_minmax<<<148 * 4, 256, 0, s>>>(d->d_in.p, n, mm);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(d->h_small.p, mm, 6 * sizeof(int), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    float mn[3], mx[3];
    for (int k = 0; k < 3; ++k) {
        int a = d->h_small.p[k], b = d->h_small.p[3 + k];
        a = a >= 0 ? a : a ^ 0x7fffffff;
        b = b >= 0 ? b : b ^ 0x7fffffff;
        memcpy(&mn[k], &a, 4);
        memcpy(&mx[k], &b, 4);
    }
    d->n_out = 0;
    if (!(mn[0] <= mx[0])) return B200_OK;  // no finite point: empty output
    Grid g;
    g.inv_leaf = 1.0f / leaf;
    // The product of the extents is taken in integers: the last leaf index is cells - 1 and the sentinel is cells, so a
    // product rounded in double (above 2^53) can make the max-corner leaf equal the sentinel and drop it.
    unsigned long long cells = 1;
    for (int k = 0; k < 3; ++k) {
        const float lo = std::floor(mn[k] * g.inv_leaf), hi = std::floor(mx[k] * g.inv_leaf);
        if (!(std::fabs(lo) < 4.0e18f && std::fabs(hi) < 4.0e18f)) B200_FAIL(B200_ERR_RANGE, "leaf size too small for the cloud extent");
        g.min_b[k] = (long long)lo;
        g.div_b[k] = (long long)hi - g.min_b[k] + 1;
        if (__builtin_mul_overflow(cells, (unsigned long long)g.div_b[k], &cells) || cells > 9000000000000000000ull)
            B200_FAIL(B200_ERR_RANGE, "leaf size too small for the cloud extent");
    }
    const unsigned long long sentinel = cells;
    int end_bit = 1;
    while (end_bit < 64 && (1ull << end_bit) <= cells) ++end_bit;
    CUDA_TRY(d->k_in.reserve(n)); CUDA_TRY(d->k_out.reserve(n)); CUDA_TRY(d->k_uniq.reserve(n));
    CUDA_TRY(d->v_in.reserve(n)); CUDA_TRY(d->v_out.reserve(n)); CUDA_TRY(d->run_cnt.reserve(n)); CUDA_TRY(d->run_off.reserve(n));
    CUDA_TRY(d->d_out.reserve(n)); CUDA_TRY(d->d_cmp.reserve(n)); CUDA_TRY(d->d_cnt.reserve(n)); CUDA_TRY(d->d_cnt_cmp.reserve(n));
    CUDA_TRY(d->keep.reserve(n));
    const int nb = (int)((n + 255) / 256);
    k_keys<<<nb, 256, 0, s>>>(d->d_in.p, (int)n, g, sentinel, d->k_in.p, d->v_in.p);
    CUDA_TRY(cudaGetLastError());
    int32_t* d_nruns = d->d_small.p + 8;
    int32_t* d_nsel = d->d_small.p + 9;
    size_t t1 = 0, t2 = 0, t3 = 0, t4 = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, t1, d->k_in.p, d->k_out.p, d->v_in.p, d->v_out.p, (int)n, 0, end_bit, s));
    CUDA_TRY(cub::DeviceRunLengthEncode::Encode(nullptr, t2, d->k_out.p, d->k_uniq.p, d->run_cnt.p, d_nruns, (int)n, s));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, t3, d->run_cnt.p, d->run_off.p, (int)n, s));
    CUDA_TRY(cub::DeviceSelect::Flagged(nullptr, t4, d->d_out.p, d->keep.p, d->d_cmp.p, d_nsel, (int)n, s));
    const size_t tmp = std::max(std::max(t1, t2), std::max(t3, t4));
    CUDA_TRY(d->cub_tmp.reserve(tmp));
    size_t tt = tmp;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(d->cub_tmp.p, tt, d->k_in.p, d->k_out.p, d->v_in.p, d->v_out.p, (int)n, 0, end_bit, s));
    tt = tmp;
    CUDA_TRY(cub::DeviceRunLengthEncode::Encode(d->cub_tmp.p, tt, d->k_out.p, d->k_uniq.p, d->run_cnt.p, d_nruns, (int)n, s));
    tt = tmp;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(d->cub_tmp.p, tt, d->run_cnt.p, d->run_off.p, (int)n, s));
    k_centroids<<<nb, 256, 0, s>>>(d->d_in.p, d->v_out.p, d->k_uniq.p, d->run_off.p, d->run_cnt.p, d_nruns, sentinel, min_points, d->d_out.p,
                                   d->d_cnt.p, d->keep.p);
    // runs beyond nruns carry stale keep flags: compact only the first nruns entries
    CUDA_TRY(cudaMemcpyAsync(d->h_small.p, d_nruns, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    const int nruns = d->h_small.p[0];
    tt = tmp;
    CUDA_TRY(cub::DeviceSelect::Flagged(d->cub_tmp.p, tt, d->d_out.p, d->keep.p, d->d_cmp.p, d_nsel, nruns, s));
    tt = tmp;
    CUDA_TRY(cub::DeviceSelect::Flagged(d->cub_tmp.p, tt, d->d_cnt.p, d->keep.p, d->d_cnt_cmp.p, d_nsel, nruns, s));
    LAUNCH_COUNT(4);
    CUDA_TRY(cudaEventRecord(d->ev1, s));
    CUDA_TRY(cudaMemcpyAsync(d->h_small.p, d_nsel, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
    d->n_out = d->h_small.p[0];
    cudaEventElapsedTime(&d->last_ms, d->ev0, d->ev1);
    return B200_OK;
}

extern "C" {

/* ---- scan downsample ---- */
int32_t b200_downsampler_create(int32_t device, b200_downsampler** out) {
    if (!out) B200_FAIL(B200_ERR_ARG, "null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) B200_FAIL(B200_ERR_CUDA, "no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) B200_FAIL(B200_ERR_ARG, "bad device ordinal");
    b200_downsampler* d = new b200_downsampler();
    d->device = device;
    CUDA_SET_DEVICE(device);
    CUDA_TRY(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreate(&d->ev0));
    CUDA_TRY(cudaEventCreate(&d->ev1));
    CUDA_TRY(d->d_small.reserve(16));
    CUDA_TRY(d->h_small.reserve(16));
    *out = d;
    return B200_OK;
}
int32_t b200_downsampler_destroy(b200_downsampler* d) {
    if (!d) return B200_OK;
    cudaSetDevice(d->device);
    if (d->stream) cudaStreamSynchronize(d->stream);
    d->d_in.release(); d->d_out.release(); d->d_cmp.release(); d->k_in.release(); d->k_out.release(); d->k_uniq.release();
    d->v_in.release(); d->v_out.release(); d->run_cnt.release(); d->run_off.release(); d->d_small.release(); d->d_cnt.release();
    d->d_cnt_cmp.release(); d->keep.release(); d->cub_tmp.release(); d->h_stage.release(); d->h_small.release();
    d->d_raw.release(); d->u_keys_in.release(); d->u_keys_out.release(); d->u_vals_in.release(); d->u_vals_out.release();
    d->d_poses.release(); d->h_poses.release();
    if (d->ev0) cudaEventDestroy(d->ev0);
    if (d->ev1) cudaEventDestroy(d->ev1);
    if (d->stream) cudaStreamDestroy(d->stream);
    delete d;
    return B200_OK;
}
/* pcl::VoxelGrid::filter (setLeafSize(leaf, leaf, leaf), setMinimumPointsNumberPerVoxel(min_points)).  Records are
 * x, y, z[, intensity] floats at stride_bytes (>= 16: the 4th float is averaged too).  out_xyzi: 4 floats per voxel in
 * ascending leaf-index order, out_count: points per voxel (either may be NULL); *n_out = number of voxels. */
int32_t b200_voxel_downsample(b200_downsampler* d, const float* xyzi, int64_t n, int64_t stride, float leaf, int32_t min_points, float* out_xyzi,
                              int32_t* out_count, int64_t max_out, int64_t* n_out) {
    if (!d || !xyzi || n < 1 || stride < 12 || !(leaf > 0.f) || min_points < 0 || n > (int64_t)0x7fffff00) B200_FAIL(B200_ERR_ARG, "bad argument");
    CUDA_SET_DEVICE(d->device);
    d->n_staged = 0;  // d_in is about to hold this cloud: an undistorted scan staged there is gone
    CUDA_TRY(d->h_stage.reserve(n));
    CUDA_TRY(d->d_in.reserve(n));
    const char* src = (const char*)xyzi;
    for (int64_t i = 0; i < n; ++i) {
        const float* p = (const float*)(src + i * stride);
        d->h_stage.p[i] = make_float4(p[0], p[1], p[2], stride >= 16 ? p[3] : 0.0f);
    }
    CUDA_TRY(cudaMemcpyAsync(d->d_in.p, d->h_stage.p, n * sizeof(float4), cudaMemcpyHostToDevice, d->stream));
    int32_t rc = downsample_run(d, n, leaf, min_points);
    if (rc) return rc;
    if (n_out) *n_out = d->n_out;
    const int64_t m = std::min<int64_t>(d->n_out, max_out);
    if (m > 0 && out_xyzi) CUDA_TRY(cudaMemcpyAsync(out_xyzi, d->d_cmp.p, m * sizeof(float4), cudaMemcpyDeviceToHost, d->stream));
    if (m > 0 && out_count) CUDA_TRY(cudaMemcpyAsync(out_count, d->d_cnt_cmp.p, m * sizeof(int32_t), cudaMemcpyDeviceToHost, d->stream));
    CUDA_TRY(cudaStreamSynchronize(d->stream));
    return B200_OK;
}
/* ImuProcess::UndistortPcl, backward half (jueying_lio/include/imu_processing.hpp:175-177,247-284): sorts the raw scan by
 * its per-point time offset and moves every point to the end-of-scan frame.  Records are floats at stride_bytes: x y z
 * first, the time offset in ms at float index time_index (pcl curvature: 9 in PointXYZINormal), intensity at
 * intensity_index (< 0: none).  poses22: K x 22 doubles {offset_time, acc, gyr, vel, pos, rot(9, row-major)} = IMUpose_ of
 * the forward propagation; x_end26: the state after the last predict.  The result stays on the device ("staged") for
 * b200_voxel_downsample_staged; out_xyzi (n x 4) / out_order (n source indices) are optional host copies. */
int32_t b200_scan_undistort(b200_downsampler* d, const float* points, int64_t n, int64_t stride, int32_t time_index, int32_t intensity_index,
                            const double* poses22, int32_t K, const double* x_end26, float* out_xyzi, int32_t* out_order) {
    if (!d || !points || n < 1 || stride < 16 || (stride & 3) || time_index < 3 || time_index * 4 >= stride || intensity_index * 4 >= stride ||
        !poses22 || K < 1 || K > 4096 || !x_end26 || n > (int64_t)0x3fffff00)
        B200_FAIL(B200_ERR_ARG, "bad argument");
    using namespace vox;
    CUDA_SET_DEVICE(d->device);
    cudaStream_t s = d->stream;
    const int sf = (int)(stride / 4);
    CUDA_TRY(d->d_raw.reserve((size_t)n * sf));
    CUDA_TRY(d->d_in.reserve(n));
    CUDA_TRY(d->u_keys_in.reserve(n)); CUDA_TRY(d->u_keys_out.reserve(n)); CUDA_TRY(d->u_vals_in.reserve(n)); CUDA_TRY(d->u_vals_out.reserve(n));
    CUDA_TRY(d->d_poses.reserve((size_t)K * 22 + 32)); CUDA_TRY(d->h_poses.reserve((size_t)K * 22 + 32));
    memcpy(d->h_poses.p, poses22, (size_t)K * 22 * sizeof(double));
    memcpy(d->h_poses.p + (size_t)K * 22, x_end26, 26 * sizeof(double));
    CUDA_TRY(cudaMemcpyAsync(d->d_poses.p, d->h_poses.p, ((size_t)K * 22 + 26) * sizeof(double), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d->d_raw.p, points, (size_t)n * stride, cudaMemcpyHostToDevice, s));  // raw records, one copy
    CUDA_TRY(cudaEventRecord(d->ev0, s));
    const int nb = (int)((n + 255) / 256);
    k_und_keys<<<nb, 256, 0, s>>>(d->d_raw.p, (int)n, sf, time_index, d->u_keys_in.p, d->u_vals_in.p);
    size_t tmp = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp, d->u_keys_in.p, d->u_keys_out.p, d->u_vals_in.p, d->u_vals_out.p, (int)n, 0, 32, s));
    CUDA_TRY(d->cub_tmp.reserve(tmp));
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(d->cub_tmp.p, tmp, d->u_keys_in.p, d->u_keys_out.p, d->u_vals_in.p, d->u_vals_out.p, (int)n, 0, 32, s));
    k_undistort<<<nb, 256, 0, s>>>(d->d_raw.p, d->u_vals_out.p, (int)n, sf, time_index, intensity_index, (const ImuPose*)d->d_poses.p, K,
                                   d->d_poses.p + (size_t)K * 22, d->d_in.p);
    LAUNCH_COUNT(2);
    CUDA_TRY(cudaEventRecord(d->ev1, s));
    if (out_xyzi) CUDA_TRY(cudaMemcpyAsync(out_xyzi, d->d_in.p, n * sizeof(float4), cudaMemcpyDeviceToHost, s));
    if (out_order) CUDA_TRY(cudaMemcpyAsync(out_order, d->u_vals_out.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
    cudaEventElapsedTime(&d->last_ms, d->ev0, d->ev1);
    d->n_staged = n;
    return B200_OK;
}
/* pcl::VoxelGrid::filter on the points staged by b200_scan_undistort (no host round trip in between); a host-side
 * b200_voxel_downsample since then has overwritten them, and this returns B200_ERR_ARG */
int32_t b200_voxel_downsample_staged(b200_downsampler* d, float leaf, int32_t min_points, int64_t* n_out) {
    if (!d || !(leaf > 0.f) || min_points < 0) B200_FAIL(B200_ERR_ARG, "bad argument");
    if (d->n_staged < 1) B200_FAIL(B200_ERR_ARG, "nothing staged");
    CUDA_SET_DEVICE(d->device);
    int32_t rc = downsample_run(d, d->n_staged, leaf, min_points);
    if (rc) return rc;
    if (n_out) *n_out = d->n_out;
    return B200_OK;
}
/* device view of the last result: float4 (x, y, z, intensity) per voxel - feeds b200_iekf_update_device without a host trip */
const void* b200_downsampler_device_points(b200_downsampler* d, int64_t* n) {
    if (!d) return nullptr;
    if (n) *n = d->n_out;
    return d->d_cmp.p;
}
float b200_downsampler_last_ms(b200_downsampler* d) { return d ? d->last_ms : 0.f; }

/* ---- map builder ---- */
int32_t b200_mapbuild_create(float leaf, uint64_t capacity_voxels, int32_t device, b200_mapbuild** out) {
    if (!out) B200_FAIL(B200_ERR_ARG, "null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) B200_FAIL(B200_ERR_CUDA, "no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) B200_FAIL(B200_ERR_ARG, "bad device ordinal");
    b200_mapbuild* h = new b200_mapbuild();
    int32_t rc = h->b.init(leaf, capacity_voxels, device);
    if (rc) { h->b.destroy(); delete h; return rc; }
    *out = h;
    return B200_OK;
}
int32_t b200_mapbuild_destroy(b200_mapbuild* h) {
    if (!h) return B200_OK;
    h->b.destroy();
    delete h;
    return B200_OK;
}
/* one keyframe: records x, y, z, intensity at stride_bytes (frames/<i>.pcd, pcl::PointXYZI), pose7 = x y z qw qx qy qz
 * (one line of poses.txt).  Asynchronous: returns once the copy and the kernel are queued. */
int32_t b200_mapbuild_add_keyframe(b200_mapbuild* h, const float* xyzi, int64_t n, int64_t stride, const double* pose7) {
    if (!h || !xyzi || !pose7 || n < 1 || stride < 12) B200_FAIL(B200_ERR_ARG, "bad argument");
    vox::Builder& b = h->b;
    CUDA_SET_DEVICE(b.device);
    // three staging slots (pinned host + device) used round robin: packing keyframe i+1 on the host overlaps the copy and the
    // accumulation of keyframe i; a slot is reused only after the kernel that read it has finished (its event)
    const int slot = (int)(b.host_frames % vox::Builder::NSTAGE);
    ++b.host_frames;
    if (!b.stage_ev[slot]) CUDA_TRY(cudaEventCreateWithFlags(&b.stage_ev[slot], cudaEventDisableTiming));
    else CUDA_TRY(cudaEventSynchronize(b.stage_ev[slot]));
    CUDA_TRY(b.stage_h[slot].reserve(n));
    CUDA_TRY(b.stage_d[slot].reserve(n));
    float4* dst = b.stage_h[slot].p;
    const char* src = (const char*)xyzi;
    if (stride == 16) memcpy(dst, src, (size_t)n * 16);  // already x y z intensity records
    else
        for (int64_t i = 0; i < n; ++i) {
            const float* p = (const float*)(src + i * stride);
            dst[i] = make_float4(p[0], p[1], p[2], stride >= 16 ? p[3] : 0.0f);
        }
    CUDA_TRY(cudaMemcpyAsync(b.stage_d[slot].p, dst, n * sizeof(float4), cudaMemcpyHostToDevice, b.stream));
    int32_t rc = b.add_device(b.stage_d[slot].p, n, pose7);
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(b.stage_ev[slot], b.stream));
    return B200_OK;
}
/* same with the keyframe already on the device as float4 (x, y, z, intensity) */
int32_t b200_mapbuild_add_keyframe_device(b200_mapbuild* h, const void* d_xyzi_float4, int64_t n, const double* pose7) {
    if (!h || !d_xyzi_float4 || !pose7 || n < 1) B200_FAIL(B200_ERR_ARG, "bad argument");
    return h->b.add_device((const float4*)d_xyzi_float4, n, pose7);
}
int32_t b200_mapbuild_add_keyframes_device(b200_mapbuild* h, const void* const* d_xyzi_float4, const int64_t* n, const double* poses7, int64_t count) {
    if (!h || !d_xyzi_float4 || !n || !poses7 || count < 1) B200_FAIL(B200_ERR_ARG, "bad argument");
    for (int64_t i = 0; i < count; ++i)
        if (!d_xyzi_float4[i] || n[i] < 1) B200_FAIL(B200_ERR_ARG, "bad keyframe in batch");
    return h->b.add_device_batch(d_xyzi_float4, n, poses7, count);
}
/* waits for the queued keyframes; number of voxels held by this rank */
int64_t b200_mapbuild_num_voxels(b200_mapbuild* h) {
    if (!h) return 0;
    if (h->b.check() < 0) return -1;
    return (int64_t)h->b.h_ctr.p[0];
}
/* Exchange of partial voxel sums between the ranks of `comm`: afterwards each voxel lives on exactly one rank
 * (owner = hash(key) mod nranks) with the sums of all ranks.  Collective; no-op for a single rank. */
int32_t b200_mapbuild_merge(b200_comm* comm, b200_mapbuild* h) {
    if (!h) B200_FAIL(B200_ERR_ARG, "null handle");
    if (!comm || comm->nranks < 2) {  // nothing to exchange; report the builder's errors like a multi-rank merge does
        CUDA_SET_DEVICE(h->b.device);
        return h->b.check();
    }
    using namespace vox;
    Builder& b = h->b;
    CUDA_SET_DEVICE(b.device);
    int32_t rc = b.check();
    if (rc) return rc;
    const int R = comm->nranks;
    const uint32_t T = b.tab.mask + 1;
    const int64_t m = b.h_ctr.p[0];
    const auto t_merge0 = std::chrono::steady_clock::now();
    CUDA_TRY(b.d_counts.reserve(2 * (size_t)R + (size_t)R * R));
    CUDA_TRY(b.h_counts.reserve((size_t)R * R + 2 * R));
    unsigned long long* d_cnt = b.d_counts.p;           // [R] my records per owner
    unsigned long long* d_cursor = b.d_counts.p + R;    // [R]
    unsigned long long* d_all = b.d_counts.p + 2 * R;   // [R][R] counts of every rank
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, R * sizeof(unsigned long long), b.stream));
    k_owner_count<<<(T + 255) / 256, 256, 0, b.stream>>>(b.tab, R, d_cnt);
    NCCL_TRY(comm, comm->AllGather(d_cnt, d_all, R, ncclUint64, comm->comm, b.stream));
    CUDA_TRY(cudaMemcpyAsync(b.h_counts.p, d_all, (size_t)R * R * sizeof(unsigned long long), cudaMemcpyDeviceToHost, b.stream));
    CUDA_TRY(cudaStreamSynchronize(b.stream));
    const double t_count = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_merge0).count();
    const bool timing = getenv("B200_TIMING") != nullptr;
    double t_alloc = 0, t_scatter = 0, t_xchg = 0, t_clear = 0;
    auto lap = [&](double& dst) {  // profiling only: drains the stream
        if (!timing) return;
        cudaStreamSynchronize(b.stream);
        dst = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_merge0).count();
    };
    const unsigned long long* all = b.h_counts.p;  // all[src * R + dst]
    std::vector<unsigned long long> send_off(R + 1, 0), recv_off(R + 1, 0);
    for (int r = 0; r < R; ++r) {
        send_off[r + 1] = send_off[r] + all[(size_t)comm->rank * R + r];
        recv_off[r + 1] = recv_off[r] + all[(size_t)r * R + comm->rank];
    }
    // exchange buffers from the stream-ordered pool (kept by the pool between merges: a cudaMalloc of 2 x 200 MB here cost
    // 3.5 - 36 ms and a device-wide synchronisation)
    {
        static bool pool_set[64] = {};
        if (b.device < 64 && !pool_set[b.device]) {
            cudaMemPool_t pool;
            unsigned long long keep = ~0ull;
            if (cudaDeviceGetDefaultMemPool(&pool, b.device) == cudaSuccess) cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
            pool_set[b.device] = true;
        }
    }
    Xfer *d_send = nullptr, *d_recv = nullptr;
    CUDA_TRY(cudaMallocAsync((void**)&d_send, std::max<size_t>(send_off[R], 1) * sizeof(Xfer), b.stream));
    CUDA_TRY(cudaMallocAsync((void**)&d_recv, std::max<size_t>(recv_off[R], 1) * sizeof(Xfer), b.stream));
    lap(t_alloc);
    unsigned long long* h_cur = b.h_counts.p + (size_t)R * R;
    for (int r = 0; r < R; ++r) h_cur[r] = send_off[r];
    CUDA_TRY(cudaMemcpyAsync(d_cursor, h_cur, R * sizeof(unsigned long long), cudaMemcpyHostToDevice, b.stream));
    k_owner_scatter<<<(T + 255) / 256, 256, 0, b.stream>>>(b.tab, R, d_cursor, d_send);
    lap(t_scatter);
    CUDA_TRY(cudaEventRecord(b.ev0, b.stream));
    NCCL_TRY(comm, comm->GroupStart());
    for (int r = 0; r < R; ++r) {
        const size_t ns = (size_t)(send_off[r + 1] - send_off[r]) * sizeof(Xfer), nr = (size_t)(recv_off[r + 1] - recv_off[r]) * sizeof(Xfer);
        if (ns) NCCL_TRY(comm, comm->Send(d_send + send_off[r], ns, ncclChar, r, comm->comm, b.stream));
        if (nr) NCCL_TRY(comm, comm->Recv(d_recv + recv_off[r], nr, ncclChar, r, comm->comm, b.stream));
    }
    NCCL_TRY(comm, comm->GroupEnd());
    CUDA_TRY(cudaEventRecord(b.ev1, b.stream));
    lap(t_xchg);
    // rebuild the table from what this rank owns
    k_table_clear<<<(T + 255) / 256, 256, 0, b.stream>>>(b.tab);
    lap(t_clear);
    CUDA_TRY(cudaMemsetAsync(b.d_ctr, 0, 8 * sizeof(unsigned int), b.stream));
    const int64_t mr = (int64_t)recv_off[R];
    if (mr) k_merge_records<<<(unsigned)((mr + 255) / 256), 256, 0, b.stream>>>(d_recv, mr, b.tab, b.d_ctr, (unsigned int)b.capacity, b.d_ctr + 1);
    cudaFreeAsync(d_send, b.stream);
    cudaFreeAsync(d_recv, b.stream);
    LAUNCH_COUNT(4);
    b.n_sorted = -1;
    rc = b.check();
    cudaEventElapsedTime(&b.last_ms, b.ev0, b.ev1);
    if (getenv("B200_TIMING")) {
        const double t_end = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_merge0).count();
        fprintf(stderr, "[b200_mapbuild_merge] rank %d: %lld voxels, table %u slots, %llu out / %llu in; cumulative ms: count+allgather %.3f, buffers %.3f, "
                        "scatter %.3f, exchange %.3f, clear %.3f, rebuild+check %.3f (NCCL events %.3f)\n", comm->rank, (long long)m, T,
                (unsigned long long)send_off[R], (unsigned long long)recv_off[R], t_count, t_alloc, t_scatter, t_xchg, t_clear, t_end, b.last_ms);
    }
    return rc;
}
float b200_mapbuild_last_exchange_ms(b200_mapbuild* h) { return h ? h->b.last_ms : 0.f; }
/* Centroids of the voxels this rank holds, ascending voxel order (z, then y, then x cell = VoxelGrid's leaf order):
 * out_xyzi 4 floats per voxel, out_count points per voxel (may be NULL); returns the number of voxels (<= max written). */
int64_t b200_mapbuild_extract(b200_mapbuild* h, float* out_xyzi, int32_t* out_count, int64_t max_out) {
    if (!h) return -1;
    vox::Builder& b = h->b;
    if (cudaSetDevice(b.device) != cudaSuccess) return -1;
    if (b.n_sorted < 0 && b.sort_slots() != B200_OK) return -1;
    const int64_t m = b.n_sorted;
    const int64_t w = std::min<int64_t>(m, max_out);
    if (w > 0 && out_xyzi) {
        if (b.d_out.reserve(m) != cudaSuccess || b.d_cnt.reserve(m) != cudaSuccess) return -1;
        vox::k_extract<<<(unsigned)((m + 255) / 256), 256, 0, b.stream>>>(b.tab, (double)b.leaf, b.d_slots2.p, m, b.d_out.p, b.d_cnt.p);
        LAUNCH_COUNT(1);
        cudaMemcpyAsync(out_xyzi, b.d_out.p, w * sizeof(float4), cudaMemcpyDeviceToHost, b.stream);
        if (out_count) cudaMemcpyAsync(out_count, b.d_cnt.p, w * sizeof(int32_t), cudaMemcpyDeviceToHost, b.stream);
        if (cudaStreamSynchronize(b.stream) != cudaSuccess) return -1;
    }
    return m;
}

}  // extern "C"
